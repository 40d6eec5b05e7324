// libb200mdm.so -- C-ABI engine (see include/b200mdm.h for the contract and the reference lines each entry
// point replaces).  Host side: weight store + repack, TMA descriptor set-up, per-(B,T) workspace, launch
// sequences for one denoiser forward / one sampler step, and the whole-loop driver (one CUDA graph of a single
// step, replayed; per-step scalars are read from device tables indexed by a device-side step counter so the
// graph never changes).
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/b200mdm.h"
#include "attention_tc.cuh"
#include "epilogues.cuh"
#include "gemm.cuh"
#include "gemm2.cuh"
#include "gemm2w.cuh"
#include "gemm_ln.cuh"
#include "postprocess.cuh"
#include "qkv_attn.cuh"
#include "kernels.cuh"
#include "target_embed.cuh"

using namespace b200;

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                               \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return fail(B200MDM_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define TRY(expr)            \
  do {                       \
    int _r = (expr);         \
    if (_r != B200MDM_OK) return _r; \
  } while (0)

// ------------------------------------------------------------------------------------------------ TMA maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int resolve_driver() {
  if (g_encode) return B200MDM_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(B200MDM_ECUDA, "cuTensorMapEncodeTiled not available");
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  return B200MDM_OK;
}
// fp16 matrix [rows, cols] with leading dimension ld (elements); box = box_rows x 64 columns, 128-byte swizzle.
// elem_bytes 2 = fp16, 4 = fp32; the box is always 128 bytes wide (64 fp16 / 32 fp32 columns) x box_rows.
static int make_map_t(CUtensorMap* m, const void* ptr, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_rows) {
  TRY(resolve_driver());
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld * elem_bytes) % 16) return fail(B200MDM_EINVAL, "TMA operand misaligned");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * elem_bytes};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / elem_bytes), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200MDM_ECUDA, "cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
  return B200MDM_OK;
}
static int make_map(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  return make_map_t(m, ptr, 2, rows, cols, ld, box_rows);
}
// fp16 tensor viewed [n][rows][cols] (cols contiguous, row pitch ld elements, sample pitch rows*ld); box {64, box_rows, 1}.
// The middle dimension is bounded per sample, so tiles that run past the last token of a sample are zero-filled
// (loads) / clipped (stores) instead of touching the next sample.
static int make_map_3d(CUtensorMap* m, const void* ptr, uint64_t n, uint64_t rows, uint64_t cols, uint64_t ld,
                       uint32_t box_rows) {
  TRY(resolve_driver());
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld * 2) % 16) return fail(B200MDM_EINVAL, "TMA operand misaligned");
  cuuint64_t gdim[3] = {cols, rows, n};
  cuuint64_t gstr[2] = {ld * 2, rows * ld * 2};
  cuuint32_t box[3] = {64, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200MDM_ECUDA, "cuTensorMapEncodeTiled(3d) failed (%d)", static_cast<int>(r));
  return B200MDM_OK;
}

// Residual stream fp16 [rows, 2d] = [hi | lo]: box {32 cols, 32 rows} with 64-byte rows and the 64-byte swizzle; an
// epilogue chunk of 32 columns moves one such box from the hi half and one from the lo half.
static int make_map_res(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t d) {
  TRY(resolve_driver());
  if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail(B200MDM_EINVAL, "TMA operand misaligned");
  cuuint64_t gdim[2] = {2 * d, rows};
  cuuint64_t gstr[1] = {d * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200MDM_ECUDA, "cuTensorMapEncodeTiled(residual) failed (%d)", static_cast<int>(r));
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ engine
struct Tensor32 {
  float* dev = nullptr;
  std::vector<int64_t> shape;
  size_t numel = 0;
};

struct LayerW {
  __half *wqkv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;
  const float *bqkv, *bo, *b1, *b2, *g1, *be1, *g2, *be2;
  CUtensorMap m_wqkv, m_wo, m_w1, m_w2;   // box 128 rows: each CTA of a pair stages half of a 256-row W tile
  CUtensorMap m_wqkv_64;                  // box 64 rows: the V half-tiles of the fused QKV + attention kernel
  CUtensorMap m_wo_256, m_w2_256;         // box 256 rows: residual+LayerNorm kernel (each CTA owns 256 output columns)
  // trans_dec only: cross-attention (multihead_attn) projections and the third LayerNorm
  __half *wq_c = nullptr, *wo_c = nullptr;           // (the K/V rows of all layers live in engine->wkv_all)
  const float *bq_c = nullptr, *bo_c = nullptr, *g3 = nullptr, *be3 = nullptr;
  CUtensorMap m_wq_c, m_wo_c_256;
};

struct GraphKey {
  int mode = -1, B = 0, T = 0, flags = 0;
  const void *pred = nullptr, *imask = nullptr, *imotion = nullptr;
  bool operator==(const GraphKey& o) const {
    return mode == o.mode && B == o.B && T == o.T && flags == o.flags && pred == o.pred && imask == o.imask &&
           imotion == o.imotion;
  }
};

// Everything sized by (batch, nframes, CFG halves): activations, their TMA maps, the conditioning rows and the captured
// step graph (whose kernel parameters are these very pointers).  The engine keeps the workspace in use as its own
// base-class fields and parks the others in a small pool, so callers that alternate between shapes (the evaluation
// loader: 32 <-> 32 x mm_num_repeats, comp_v6_model_dataset.py:148-256) neither re-allocate nor re-capture.
struct Workspace {
  int B = 0, T = 0, S = 0, halves = 1, Bp = 0, M = 0, MB = 0;
  __half *xin16 = nullptr, *hres = nullptr, *qkv16 = nullptr, *att16 = nullptr, *ffn16 = nullptr, *g16 = nullptr;
  float *tok0 = nullptr, *condproj = nullptr, *proj = nullptr, *scale = nullptr, *x_work = nullptr, *eps_buf = nullptr;
  int *kvlen = nullptr, *tvec = nullptr, *action = nullptr;
  CUtensorMap m_xin, m_h16, m_att, m_ffn, m_g16;      // A operands (loads, box 128 rows)
  CUtensorMap m_qkv_st, m_ffn_st;                      // epilogue slabs (box 32 rows x 128 bytes)
  CUtensorMap m_res;                                   // residual stream [hi | lo] (make_map_res)
  CUtensorMap m_att_q, m_att_kv, m_att_o;             // tcgen05 attention: per-sample 3-D views of qkv16 / att16
  CUtensorMap m_h3;                                    // fused QKV+attention: per-sample A tiles of the stream's hi half
  CUtensorMap m_res_c, m_res_u;                        // per-CFG-half views of the residual stream (embedding epilogue)
  float* pe_bias = nullptr;
  bool cond_set = false;
  // trans_dec (DiP): prefix frames + text-token memory
  int Mt = 0;
  float *encperm = nullptr, *memtok = nullptr, *memproj = nullptr;   // [B*Mt, cond_dim], [B*Mt, d], [Bp*Mt, d]
  __half *mem16 = nullptr, *qc16 = nullptr, *kvc16 = nullptr;        // [Bp*Mt, d], [M, d], [Bp*Mt, 2d]
  unsigned char* memmask = nullptr;                                   // [Bp, Mt] 1 = padding
  CUtensorMap m_mem, m_qc_st, m_kvc_st;
  bool prefix_set = false;
  // captured step graph of this workspace
  cudaGraphExec_t graph_exec = nullptr;
  GraphKey graph_key;
  int graph_kernels = 0;
  unsigned long long last_use = 0;
};

struct b200mdm_engine : Workspace {
  b200mdm_config cfg;
  int d, ff, L, H, JF, Kp_in, N_out_pad;
  int num_sms = 148;
  std::map<std::string, Tensor32> store;
  bool finalized = false;
  // repacked weights
  __half *w_in3 = nullptr, *w_out3 = nullptr;
  CUtensorMap m_win, m_wout;
  std::vector<LayerW> layers;
  const float *b_in = nullptr, *b_out = nullptr, *pe = nullptr, *w_txt = nullptr, *b_txt = nullptr, *act_emb = nullptr;
  float *temb_hidden = nullptr, *temb_table = nullptr;
  // trans_dec: key/value projection rows of the cross-attention of ALL layers, [L * 2d, d] fp16 + bias [L * 2d]: the text
  // memory is the same for every layer, so one GEMM per step projects it for all of them
  __half* wkv_all = nullptr;
  float* bkv_all = nullptr;
  CUtensorMap m_wkv_all;
  // schedule (device tables are allocated once at `sched_cap` rows: the step graphs hold these pointers)
  float* sched = nullptr;
  int* tmap = nullptr;
  int n_steps = 0, sched_cap = 0;
  // parked workspaces (see Workspace)
  std::vector<Workspace> pool;
  unsigned long long use_clock = 0;
  // host staging for b200mdm_set_cond* (kept alive until the next call: no stream synchronisation needed)
  std::vector<int> h_kv, h_action;
  std::vector<unsigned char> h_mask;
  // trans_dec (DiP)
  bool dec = false;
  int ctx = 0, s_off = 1;
  int kw = 1;   // 2: fp16 activations between the layer GEMMs are [hi | lo] pairs along K (trans_dec engine)
  const unsigned char* inpaint_mask = nullptr;
  const float* inpaint_motion = nullptr;
  // in-engine noise (B200MDM_FLAG_PHILOX_NOISE): counter-based Philox4x32-10 keyed by (seed, schedule index, global sample)
  unsigned long long noise_seed = 0;
  long long noise_sample_base = 0;
  // loop machinery
  StepState* state = nullptr;   // device-side step counter + per-loop noise description, shared by every workspace
  cudaStream_t work = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  long long launches = 0;
  // target-location encoder (b200mdm_set_target): weights packed per stage as [groups, N, K] / [groups, N], buffers sized
  // for `tgt_cap` samples (they only grow), and the embedding the next set_cond* folds into its conditioning rows
  std::vector<float*> tgt_w, tgt_b;
  float* tgt_wn = nullptr;                                   // multi: w / sum(w)
  float *tgt_out = nullptr, *tgt_ha = nullptr, *tgt_hb = nullptr, *tgt_x0 = nullptr;
  int* tgt_idx = nullptr;                                    // [n counts | n x cap sample lists | cap x n validity]
  int tgt_cap = 0, tgt_batch = 0;
  bool tgt_pending = false;
  std::vector<int> h_tgt;
};

template <class T>
static int dalloc(T** p, size_t n, bool zero = false) {
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)));
  if (zero) CUDA_TRY(cudaMemset(*p, 0, n * sizeof(T)));
  return B200MDM_OK;
}
template <class T>
static void dfree(T*& p) {
  if (p) cudaFree(p);
  p = nullptr;
}

// ------------------------------------------------------------------------------------------------ launchers
template <int BN, class Epi>
static int set_gemm_attr() {
  CUDA_TRY(cudaFuncSetAttribute(gemm_f16_tcgen05<BN, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                GemmSmem<BN, Epi>::TOTAL));
  return B200MDM_OK;
}
template <class Epi>
static int set_gemm2_attr() {
  CUDA_TRY(cudaFuncSetAttribute(gemm2_f16_tcgen05<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, Gemm2Smem<Epi>::TOTAL));
  return B200MDM_OK;
}
static int init_kernel_attrs() {
  // function attributes are per device: track which ordinals have been initialised
  static unsigned long long done_mask = 0;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 64 && ((done_mask >> dev) & 1ull)) return B200MDM_OK;
  TRY((set_gemm_attr<128, EpiBiasF16<false>>()));
  TRY((set_gemm_attr<128, EpiBiasF16<true>>()));
  TRY((set_gemm2_attr<EpiBiasF16<false>>()));
  TRY((set_gemm2_attr<EpiBiasF16<true>>()));
  TRY((set_gemm2_attr<EpiBiasF16Wide<true>>()));
  TRY((set_gemm2_attr<EpiBiasF16Global>()));
  CUDA_TRY(cudaFuncSetAttribute(gemm2w_f16_tcgen05<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Gemm2wSmem::TOTAL));
  CUDA_TRY(cudaFuncSetAttribute(gemm2w_f16_tcgen05<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Gemm2wSmem::TOTAL));
  CUDA_TRY(cudaFuncSetAttribute(gemm_resid_ln_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmLnSmem::TOTAL));
  TRY((set_gemm_attr<128, EpiEmbed>()));
  TRY((set_gemm_attr<96, EpiOutStep>()));
  CUDA_TRY(cudaFuncSetAttribute(qkv_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, QkvAttnSmem::TOTAL));
  CUDA_TRY(cudaFuncSetAttribute(attention_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                AttnTcSmem::total(ATC_MAX_KEYS)));
  CUDA_TRY(cudaFuncSetAttribute(attention_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                AttnTcSmem::total(ATC_MAX_KEYS)));
  if (dev < 64) done_mask |= 1ull << dev;
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ launches
// Kernels of the sampling step are launched with programmatic stream serialization (PDL): the next kernel's CTAs are
// scheduled as SMs drain and run their prologue (barrier init, TMEM allocation, descriptor prefetch, bias staging)
// under the tail of the current one; every kernel calls griddepcontrol.wait before it touches global data.
// B200MDM_PDL=0 in the environment restores plain stream order.
static bool g_pdl_now = false;   // set while b200mdm is enqueueing a step
static bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200MDM_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
struct PdlScope {
  PdlScope() { g_pdl_now = pdl_enabled(); }
  ~PdlScope() { g_pdl_now = false; }
};
template <class... KArgs, class... Args>
static cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = g_pdl_now ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(std::forward<Args>(args))...);
}

template <int BN, class Epi>
static int launch_gemm(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, int M, int N, int K,
                       const typename Epi::Params& p, cudaStream_t s, int num_sms) {
  if (N * 4 > GEMM_BIAS_BYTES) return fail(B200MDM_ENOTIMPL, "GEMM epilogue vectors are staged for N <= %d", GEMM_BIAS_BYTES / 4);
  const int tiles = ((M + GEMM_BLOCK_M - 1) / GEMM_BLOCK_M) * ((N + BN - 1) / BN);
  const int grid = tiles < num_sms ? tiles : num_sms;
  CUDA_TRY(launch_k(gemm_f16_tcgen05<BN, Epi>, dim3(grid), dim3(GEMM_THREADS), GemmSmem<BN, Epi>::TOTAL, s, a, b, c, M, N, K, p));
  return B200MDM_OK;
}

// CTA-pair GEMM (256 x 256 tiles): a = A map (box 128 rows), b = W map with box 128 rows (half tile per CTA)
template <class Epi, class = void> struct epi_unstaged : std::false_type {};
template <class Epi> struct epi_unstaged<Epi, std::enable_if_t<Epi::UNSTAGED>> : std::true_type {};

template <class Epi>
static int launch_gemm2(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, int M, int N, int K,
                        const typename Epi::Params& p, cudaStream_t s, int num_sms) {
  if (!epi_unstaged<Epi>::value && N * 4 > GEMM_BIAS_BYTES) return fail(B200MDM_ENOTIMPL, "GEMM epilogue vectors are staged for N <= %d", GEMM_BIAS_BYTES / 4);
  const int tiles = ((M + GEMM2_TILE_M - 1) / GEMM2_TILE_M) * ((N + GEMM2_BLOCK_N - 1) / GEMM2_BLOCK_N);
  const int max_clusters = num_sms / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  CUDA_TRY(launch_k(gemm2_f16_tcgen05<Epi>, dim3(2 * clusters), dim3(GEMM2_THREADS), Gemm2Smem<Epi>::TOTAL, s, a, b, c, M, N, K, p));
  return B200MDM_OK;
}

// W-resident CTA-pair GEMM (gemm2w.cuh): K <= 512, every column block owned by at least one cluster.
template <bool GELU>
static int launch_gemm2w(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, int M, int N, int K,
                         const float* bias, cudaStream_t s, int num_sms) {
  const int tiles_n = (N + GEMM2_BLOCK_N - 1) / GEMM2_BLOCK_N;
  const int tiles = ((M + GEMM2_TILE_M - 1) / GEMM2_TILE_M) * tiles_n;
  const int max_clusters = num_sms / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  if (K > GEMM2W_KB_MAX * GEMM_BLOCK_K || tiles_n > clusters)
    return fail(B200MDM_ENOTIMPL, "W-resident pair GEMM needs K <= %d and N <= %d", GEMM2W_KB_MAX * GEMM_BLOCK_K, clusters * GEMM2_BLOCK_N);
  typename EpiBiasF16<GELU>::Params p{bias};
  CUDA_TRY(launch_k(gemm2w_f16_tcgen05<GELU>, dim3(2 * clusters), dim3(GEMM2_THREADS), Gemm2wSmem::TOTAL, s, a, b, c, M, N, K, p));
  return B200MDM_OK;
}
// The W-resident order binds a cluster to one column block: it pays when that costs no extra round of tiles compared
// with the strided order of the streaming kernel (rounds = tiles on the busiest cluster).  B200MDM_GEMM2W=0 in the
// environment keeps the streaming kernel everywhere (A/B timing).
static bool gemm2w_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200MDM_GEMM2W");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
static bool gemm2w_pays(int M, int N, int K, int num_sms) {
  if (!gemm2w_enabled() || K > GEMM2W_KB_MAX * GEMM_BLOCK_K) return false;
  const int tiles_m = (M + GEMM2_TILE_M - 1) / GEMM2_TILE_M;
  const int tiles_n = (N + GEMM2_BLOCK_N - 1) / GEMM2_BLOCK_N;
  const int tiles = tiles_m * tiles_n;
  const int max_clusters = num_sms / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  if (tiles_n > clusters) return false;
  const int rounds_strided = (tiles + clusters - 1) / clusters;
  const int owners = clusters / tiles_n;   // clusters of the least-served column block
  const int rounds_resident = (tiles_m + owners - 1) / owners;
  return rounds_resident <= rounds_strided;
}
// out16 = fp16(act(A W^T + bias)) on CTA pairs: W-resident kernel where it pays, streaming kernel otherwise
template <bool GELU>
static int launch_gemm2_bias(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, int M, int N, int K,
                             const float* bias, cudaStream_t s, int num_sms) {
  if (gemm2w_pays(M, N, K, num_sms)) return launch_gemm2w<GELU>(a, b, c, M, N, K, bias, s, num_sms);
  typename EpiBiasF16<GELU>::Params p{bias};
  return launch_gemm2<EpiBiasF16<GELU>>(a, b, c, M, N, K, p, s, num_sms);
}

// h <- LayerNorm(h + A W^T + bias), 2-CTA cluster splitting the 512 columns, LayerNorm statistics exchanged through
// distributed shared memory (w256: W map with box 256 rows)
static int launch_gemm_resid_ln(const CUtensorMap& a, const CUtensorMap& w256, const CUtensorMap& res, int M, int K,
                                const float* bias, const float* gamma, const float* beta, cudaStream_t s, int num_sms) {
  const int tiles = (M + GEMM_BLOCK_M - 1) / GEMM_BLOCK_M;
  const int max_clusters = num_sms / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  GemmLnParams lp{bias, gamma, beta, 1e-5f};
  CUDA_TRY(launch_k(gemm_resid_ln_cluster, dim3(2 * clusters), dim3(GLN_THREADS), GemmLnSmem::TOTAL, s, a, w256, res, M, K, lp));
  return B200MDM_OK;
}

struct AttnMaps {
  CUtensorMap q, kv, o;
};
static int make_attn_maps(AttnMaps* m, const __half* qkv, __half* out, int n_samples, int S, int d, int kw = 1) {
  const int keys = (S + 15) & ~15;
  TRY(make_map_3d(&m->q, qkv, n_samples, S, 3 * d, 3 * d, 128));
  TRY(make_map_3d(&m->kv, qkv, n_samples, S, 3 * d, 3 * d, keys));
  TRY(make_map_3d(&m->o, out, n_samples, S, kw * d, kw * d, 32));   // kw = 2: [hi | lo] output rows
  return B200MDM_OK;
}
// tcgen05 kernel for sequences of up to 256 tokens (every configuration of the reference: 197 / 61 / 60)
static int launch_attention_tc(const AttnMaps& m, const int* kvlen, int n_samples, int S, int d, int H, cudaStream_t s,
                               bool wide = false) {
  if (d != H * ATC_DH) return fail(B200MDM_ENOTIMPL, "attention: head_dim must be 128");
  const int keys = (S + 15) & ~15;
  const float scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(ATC_DH));
  const dim3 grid(H, n_samples, (S + 127) / 128);
  CUDA_TRY(launch_k(wide ? attention_tc_kernel<true> : attention_tc_kernel<false>, grid, dim3(ATC_THREADS), AttnTcSmem::total(keys),
                    s, m.q, m.kv, m.o, kvlen, S, d, keys, scale_log2));
  return B200MDM_OK;
}

// fused QKV projection + attention (qkv_attn.cuh): one CTA pair per (sample, head), persistent
static int launch_qkv_attention(const CUtensorMap& h3, const CUtensorMap& w128, const CUtensorMap& w64, const CUtensorMap& o,
                                const float* bqkv, const int* kvlen, int n_samples, int S, cudaStream_t s, int num_sms) {
  if (S > 256) return fail(B200MDM_ENOTIMPL, "fused attention: at most 256 tokens per sample");
  const int items = n_samples * 4;
  const int max_clusters = num_sms / 2;
  const int clusters = items < max_clusters ? items : max_clusters;
  const float scale_log2 = 1.4426950408889634f / sqrtf(128.0f);
  CUDA_TRY(launch_k(qkv_attention_kernel, dim3(2 * clusters), dim3(QA_THREADS), QkvAttnSmem::TOTAL, s, h3, w128, w64, o, bqkv, kvlen,
                    n_samples, S, scale_log2));
  return B200MDM_OK;
}
#ifdef B200_TRACE
// Instrumented build only (lib/libb200mdm_trace.so): B200MDM_DEBUG_SKIP is a bit mask of layer kernels to leave out of the
// step (1 attention, 2 out-proj+LN, 4 FFN-up, 8 FFN-down+LN) -- the results are garbage, the loop time difference is what
// that kernel costs INSIDE the graph loop (programmatic dependent launch, L2 window), which no profiler shows.
static int debug_skip_mask() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200MDM_DEBUG_SKIP");
    v = e ? atoi(e) : 0;
  }
  return v;
}
#define B200_SKIP(bit) (debug_skip_mask() & (bit))
#else
#define B200_SKIP(bit) (0)
#endif
// The fused QKV-projection + attention kernel works on one 256-row CTA-pair tile per (sample, head) whatever the sample
// length: at S = 197 (HumanML3D) it is the fast path, at S = 61 (HumanAct12 / UESTC, 76 % padding) the separate
// projection GEMM + attention core is 40 % faster end to end (137 vs 98 motions/s on the a2m configuration).  A sample
// that fills only one CTA of the pair (S <= 128) therefore takes the unfused path.  B200MDM_FUSED_QKV=0 / 1 forces it.
static bool fused_qkv_enabled(int S) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200MDM_FUSED_QKV");
    v = !e ? 2 : (e[0] == '0' ? 0 : 1);
  }
  return v == 2 ? (S > 128 && S <= 256) : v == 1;
}

// ------------------------------------------------------------------------------------------------ API: basics
extern "C" const char* b200mdm_last_error(void) { return g_err; }
extern "C" int b200mdm_version(void) { return 1; }

extern "C" int b200mdm_create(const b200mdm_config* cfg, b200mdm_engine** out) {
  if (!cfg || !out) return fail(B200MDM_EINVAL, "null argument");
  if (cfg->arch != B200MDM_ARCH_TRANS_ENC && cfg->arch != B200MDM_ARCH_TRANS_DEC)
    return fail(B200MDM_ENOTIMPL, "arch %d: trans_enc and trans_dec are implemented", cfg->arch);
  if (cfg->arch == B200MDM_ARCH_TRANS_DEC && (cfg->cond_mode != B200MDM_COND_TEXT || cfg->context_len < 0))
    return fail(B200MDM_ENOTIMPL, "trans_dec needs text-token conditioning (BERT) and context_len >= 0");
  if (cfg->latent_dim != 512 || cfg->num_heads != 4 || cfg->ff_size % 64 || cfg->ff_size <= 0)
    return fail(B200MDM_ENOTIMPL, "kernels are specialised for latent_dim 512 / 4 heads (got %d / %d)", cfg->latent_dim,
                cfg->num_heads);
  if (cfg->num_layers <= 0 || cfg->njoints <= 0 || cfg->nfeats <= 0 || cfg->pos_embed_max_len <= 0 || cfg->temb_rows <= 0)
    return fail(B200MDM_EINVAL, "bad config");
  if (cfg->target_encoder != B200MDM_TARGET_NONE) {
    if (cfg->target_encoder < B200MDM_TARGET_SINGLE || cfg->target_encoder > B200MDM_TARGET_SPLIT)
      return fail(B200MDM_ENOTIMPL, "target_encoder %d: single (1), multi (2) and split (3) are implemented", cfg->target_encoder);
    if (cfg->n_goal_rows < 1 || cfg->n_goal_rows > 64)
      return fail(B200MDM_ENOTIMPL, "target encoder: n_goal_rows %d outside 1..64", cfg->n_goal_rows);
    if (cfg->target_encoder != B200MDM_TARGET_MULTI && cfg->target_enc_layers < 1)
      return fail(B200MDM_ENOTIMPL, "target encoder: target_enc_layers %d (>= 1 implemented)", cfg->target_enc_layers);
    if (cfg->target_encoder == B200MDM_TARGET_SPLIT && cfg->latent_dim % cfg->n_goal_rows)
      return fail(B200MDM_ENOTIMPL, "split target encoder needs latent_dim %% n_goal_rows == 0 (%d, %d)", cfg->latent_dim,
                  cfg->n_goal_rows);
  }
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(B200MDM_ECUDA, "sm_100a device required (found sm_%d%d)", prop.major, prop.minor);
  TRY(init_kernel_attrs());
  TRY(resolve_driver());
  b200mdm_engine* e = new b200mdm_engine();
  e->cfg = *cfg;
  e->d = cfg->latent_dim;
  e->ff = cfg->ff_size;
  e->L = cfg->num_layers;
  e->H = cfg->num_heads;
  e->JF = cfg->njoints * cfg->nfeats;
  e->Kp_in = (e->JF + 7) & ~7;
  e->N_out_pad = ((e->JF + 95) / 96) * 96;
  e->num_sms = prop.multiProcessorCount;
  e->layers.resize(e->L);
  e->dec = cfg->arch == B200MDM_ARCH_TRANS_DEC;
  e->ctx = e->dec ? cfg->context_len : 0;
  e->s_off = e->dec ? e->ctx : 1;
  // DiP samples with guidance 7.5 (three times the encoder's 2.5): the CFG blend multiplies every activation rounding
  // error by ~10.  Its fp16 activations are therefore kept as hi + lo pairs; at 60-token sequences the doubled K of
  // the layer GEMMs is free.
  e->kw = e->dec ? 2 : 1;
  CUDA_TRY(cudaStreamCreateWithFlags(&e->work, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming));
  TRY(dalloc(&e->state, 1, true));
  *out = e;
  return B200MDM_OK;
}

static void drop_graph(Workspace* w) {
  if (w->graph_exec) cudaGraphExecDestroy(w->graph_exec);
  w->graph_exec = nullptr;
  w->graph_key = GraphKey();
}
static void free_workspace(Workspace* w) {
  drop_graph(w);
  dfree(w->xin16); dfree(w->hres); dfree(w->qkv16); dfree(w->att16); dfree(w->ffn16); dfree(w->g16);
  dfree(w->tok0); dfree(w->condproj); dfree(w->proj); dfree(w->scale); dfree(w->x_work); dfree(w->pe_bias); dfree(w->eps_buf);
  dfree(w->kvlen); dfree(w->tvec); dfree(w->action);
  dfree(w->encperm); dfree(w->memtok); dfree(w->memproj); dfree(w->mem16); dfree(w->qc16); dfree(w->kvc16); dfree(w->memmask);
  *w = Workspace();
}
// every workspace (the one in use and the parked ones): after a weight reload or a schedule-table move their graphs
// and derived tables (pe_bias, condproj, memproj) are stale
static void free_all_workspaces(b200mdm_engine* e) {
  free_workspace(static_cast<Workspace*>(e));
  for (auto& w : e->pool) free_workspace(&w);
  e->pool.clear();
}
static void drop_all_graphs(b200mdm_engine* e) {
  drop_graph(static_cast<Workspace*>(e));
  for (auto& w : e->pool) drop_graph(&w);
}

static void free_target(b200mdm_engine* e, bool buffers) {
  for (float* p : e->tgt_w) cudaFree(p);
  for (float* p : e->tgt_b) cudaFree(p);
  e->tgt_w.clear();
  e->tgt_b.clear();
  dfree(e->tgt_wn);
  if (buffers) {
    dfree(e->tgt_out); dfree(e->tgt_ha); dfree(e->tgt_hb); dfree(e->tgt_x0); dfree(e->tgt_idx);
    e->tgt_cap = 0;
  }
  e->tgt_pending = false;
}

extern "C" int b200mdm_destroy(b200mdm_engine* e) {
  if (!e) return B200MDM_OK;
  cudaDeviceSynchronize();
  free_all_workspaces(e);
  for (auto& kv : e->store) cudaFree(kv.second.dev);
  for (auto& l : e->layers) { dfree(l.wqkv); dfree(l.wo); dfree(l.w1); dfree(l.w2); dfree(l.wq_c); dfree(l.wo_c); }
  dfree(e->w_in3); dfree(e->w_out3); dfree(e->temb_hidden); dfree(e->temb_table); dfree(e->sched); dfree(e->tmap);
  dfree(e->wkv_all); dfree(e->bkv_all);
  free_target(e, true);
  dfree(e->state);
  if (e->work) cudaStreamDestroy(e->work);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  delete e;
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ weights
// The target encoder as a chain of grouped linear stages (target_embed.cuh): stage s has `groups` matrices [N, K]; the
// state_dict name of group g's weight is name(s, g) + ".weight", its bias name(s, g) + ".bias".
struct TgtStage {
  int groups, N, K;
};
static std::vector<TgtStage> target_stages(const b200mdm_config& c) {
  const int d = c.latent_dim, n = c.n_goal_rows;
  std::vector<TgtStage> st;
  if (c.target_encoder == B200MDM_TARGET_SINGLE) {
    st.push_back({1, d, 4 * n});
    for (int l = 0; l < c.target_enc_layers; ++l) st.push_back({1, d, d});
  } else if (c.target_encoder == B200MDM_TARGET_SPLIT) {
    st.push_back({n, d / n, 4});
    for (int l = 0; l < c.target_enc_layers; ++l) st.push_back({n, d / n, d / n});
  } else if (c.target_encoder == B200MDM_TARGET_MULTI) {
    st.push_back({n, d, 3});
    st.push_back({n, d, d});
  }
  return st;
}
static std::string target_stage_name(const b200mdm_config& c, int s, int g) {
  const std::string p = "embed_target_cond.";
  if (c.target_encoder == B200MDM_TARGET_SINGLE) return p + "mlp." + std::to_string(2 * s);
  if (c.target_encoder == B200MDM_TARGET_SPLIT) return p + "mini_mlps." + std::to_string(g) + "." + std::to_string(2 * s);
  return p + "target_loc_emb." + std::to_string(g) + "." + std::to_string(2 * s);
}
static const char* kTargetRowWeights = "embed_target_cond.target_all_loc_emb.weights";

static bool known_target_name(const b200mdm_engine* e, const std::string& n) {
  if (e->cfg.target_encoder == B200MDM_TARGET_NONE || n.compare(0, 18, "embed_target_cond.") != 0) return false;
  if (e->cfg.target_encoder == B200MDM_TARGET_MULTI && n == kTargetRowWeights) return true;
  const std::vector<TgtStage> st = target_stages(e->cfg);
  for (size_t s = 0; s < st.size(); ++s)
    for (int g = 0; g < st[s].groups; ++g) {
      const std::string base = target_stage_name(e->cfg, static_cast<int>(s), g);
      if (n == base + ".weight" || n == base + ".bias") return true;
    }
  return false;
}

static bool known_weight_name(const b200mdm_engine* e, const std::string& n) {
  if (known_target_name(e, n)) return true;
  static const char* fixed[] = {"input_process.poseEmbedding.weight", "input_process.poseEmbedding.bias",
                                "embed_timestep.time_embed.0.weight", "embed_timestep.time_embed.0.bias",
                                "embed_timestep.time_embed.2.weight", "embed_timestep.time_embed.2.bias",
                                "embed_text.weight", "embed_text.bias", "embed_action.action_embedding",
                                "output_process.poseFinal.weight", "output_process.poseFinal.bias",
                                "sequence_pos_encoder.pe", "embed_timestep.sequence_pos_encoder.pe"};
  for (const char* f : fixed)
    if (n == f) return true;
  static const char* per_layer[] = {"self_attn.in_proj_weight", "self_attn.in_proj_bias", "self_attn.out_proj.weight",
                                    "self_attn.out_proj.bias", "linear1.weight", "linear1.bias", "linear2.weight",
                                    "linear2.bias", "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias",
                                    "multihead_attn.in_proj_weight", "multihead_attn.in_proj_bias",
                                    "multihead_attn.out_proj.weight", "multihead_attn.out_proj.bias", "norm3.weight", "norm3.bias"};
  const std::string pre = e->dec ? "seqTransDecoder.layers." : "seqTransEncoder.layers.";
  if (n.compare(0, pre.size(), pre) == 0) {
    size_t dot = n.find('.', pre.size());
    if (dot == std::string::npos) return false;
    int l = atoi(n.substr(pre.size(), dot - pre.size()).c_str());
    if (l < 0 || l >= e->L) return false;
    std::string rest = n.substr(dot + 1);
    for (const char* f : per_layer)
      if (rest == f) return true;
  }
  return false;
}

extern "C" int b200mdm_load_weight(b200mdm_engine* e, const char* name, const float* data, const int64_t* shape,
                                   int32_t ndim) {
  if (!e || !name || !data || !shape || ndim < 1 || ndim > 4) return fail(B200MDM_EINVAL, "bad argument");
  std::string n(name);
  if (!known_weight_name(e, n)) return fail(B200MDM_EINVAL, "unexpected state_dict key '%s'", name);
  size_t numel = 1;
  std::vector<int64_t> shp(shape, shape + ndim);
  for (int64_t s : shp) {
    if (s <= 0) return fail(B200MDM_EINVAL, "bad shape for '%s'", name);
    numel *= static_cast<size_t>(s);
  }
  Tensor32& t = e->store[n];
  if (t.dev && t.numel != numel) { cudaFree(t.dev); t.dev = nullptr; }
  if (!t.dev) TRY(dalloc(&t.dev, numel));
  t.shape = shp;
  t.numel = numel;
  CUDA_TRY(cudaMemcpy(t.dev, data, numel * sizeof(float), cudaMemcpyDefault));
  e->finalized = false;
  return B200MDM_OK;
}

static int need(b200mdm_engine* e, const std::string& name, std::initializer_list<int64_t> shape, const float** out) {
  auto it = e->store.find(name);
  if (it == e->store.end()) return fail(B200MDM_ESTATE, "missing weight '%s'", name.c_str());
  std::vector<int64_t> want(shape);
  // allow a leading singleton / trailing squeeze for the positional table [max_len, 1, d]
  size_t numel = 1;
  for (int64_t s : want) numel *= static_cast<size_t>(s);
  if (it->second.numel != numel) return fail(B200MDM_EINVAL, "weight '%s' has %zu elements, expected %zu", name.c_str(), it->second.numel, numel);
  *out = it->second.dev;
  return B200MDM_OK;
}

static int to_f16(const float* src, __half** dst, size_t n, cudaStream_t s) {
  TRY(dalloc(dst, n));
  f32_to_f16_kernel<<<512, 256, 0, s>>>(src, *dst, n);
  CUDA_TRY(cudaGetLastError());
  return B200MDM_OK;
}
// W [N, K] -> fp16 [N, kw * K]: kw = 2 repeats W along K for activations kept as [hi | lo] (trans_dec engine)
static int to_f16_k(const float* src, __half** dst, int N, int K, int kw, cudaStream_t s) {
  if (kw == 1) return to_f16(src, dst, static_cast<size_t>(N) * K, s);
  TRY(dalloc(dst, static_cast<size_t>(N) * K * 2));
  f32_to_f16_dup_kernel<<<512, 256, 0, s>>>(src, *dst, N, K);
  CUDA_TRY(cudaGetLastError());
  return B200MDM_OK;
}

// Pack every stage of the target encoder into [groups, N, K] / [groups, N] (one grouped launch per stage), and normalise
// the multi encoder's row weights.
static int finalize_target(b200mdm_engine* e, cudaStream_t s) {
  free_target(e, false);
  if (e->cfg.target_encoder == B200MDM_TARGET_NONE) return B200MDM_OK;
  const std::vector<TgtStage> st = target_stages(e->cfg);
  for (size_t k = 0; k < st.size(); ++k) {
    const TgtStage& g = st[k];
    float *w = nullptr, *b = nullptr;
    TRY(dalloc(&w, static_cast<size_t>(g.groups) * g.N * g.K));
    e->tgt_w.push_back(w);
    TRY(dalloc(&b, static_cast<size_t>(g.groups) * g.N));
    e->tgt_b.push_back(b);
    for (int j = 0; j < g.groups; ++j) {
      const std::string base = target_stage_name(e->cfg, static_cast<int>(k), j);
      const float *src_w, *src_b;
      TRY(need(e, base + ".weight", {g.N, g.K}, &src_w));
      TRY(need(e, base + ".bias", {g.N}, &src_b));
      CUDA_TRY(cudaMemcpyAsync(w + static_cast<size_t>(j) * g.N * g.K, src_w, sizeof(float) * g.N * g.K, cudaMemcpyDeviceToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(b + static_cast<size_t>(j) * g.N, src_b, sizeof(float) * g.N, cudaMemcpyDeviceToDevice, s));
    }
  }
  if (e->cfg.target_encoder == B200MDM_TARGET_MULTI) {
    const float* rw;
    TRY(need(e, kTargetRowWeights, {e->cfg.n_goal_rows}, &rw));
    TRY(dalloc(&e->tgt_wn, e->cfg.n_goal_rows));
    tgt_normalise_kernel<<<1, 1, 0, s>>>(rw, e->tgt_wn, e->cfg.n_goal_rows);
    CUDA_TRY(cudaGetLastError());
  }
  return B200MDM_OK;
}

extern "C" int b200mdm_finalize_weights(b200mdm_engine* e, void* stream) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int d = e->d, ff = e->ff, JF = e->JF;
  const float *w_in, *w_out, *t0w, *t0b, *t2w, *t2b;
  TRY(need(e, "input_process.poseEmbedding.weight", {d, JF}, &w_in));
  TRY(need(e, "input_process.poseEmbedding.bias", {d}, &e->b_in));
  TRY(need(e, "output_process.poseFinal.weight", {JF, d}, &w_out));
  TRY(need(e, "output_process.poseFinal.bias", {JF}, &e->b_out));
  TRY(need(e, "embed_timestep.time_embed.0.weight", {d, d}, &t0w));
  TRY(need(e, "embed_timestep.time_embed.0.bias", {d}, &t0b));
  TRY(need(e, "embed_timestep.time_embed.2.weight", {d, d}, &t2w));
  TRY(need(e, "embed_timestep.time_embed.2.bias", {d}, &t2b));
  TRY(need(e, "sequence_pos_encoder.pe", {e->cfg.pos_embed_max_len, d}, &e->pe));
  if (e->cfg.cond_mode == B200MDM_COND_TEXT) {
    TRY(need(e, "embed_text.weight", {d, e->cfg.cond_dim}, &e->w_txt));
    TRY(need(e, "embed_text.bias", {d}, &e->b_txt));
  } else if (e->cfg.cond_mode == B200MDM_COND_ACTION) {
    TRY(need(e, "embed_action.action_embedding", {e->cfg.num_actions, d}, &e->act_emb));
  }
  if (e->cfg.temb_rows > e->cfg.pos_embed_max_len) return fail(B200MDM_EINVAL, "temb_rows exceeds the positional table");

  // drop previous repacks; every workspace holds tables derived from the weights (pe_bias, condproj, memproj) and a
  // graph whose kernel parameters point at the old repacks: a forward that ran before this load must not leak into
  // the next one
  CUDA_TRY(cudaDeviceSynchronize());
  free_all_workspaces(e);
  for (auto& l : e->layers) { dfree(l.wqkv); dfree(l.wo); dfree(l.w1); dfree(l.w2); dfree(l.wq_c); dfree(l.wo_c); }
  dfree(e->w_in3); dfree(e->w_out3); dfree(e->temb_hidden); dfree(e->temb_table); dfree(e->wkv_all); dfree(e->bkv_all);

  // split-precision in / out projections: W' = [hi | hi | lo], zero padded
  const int Kp = e->Kp_in;
  TRY(dalloc(&e->w_in3, static_cast<size_t>(d) * 3 * Kp, true));
  split_weight_kernel<<<d, 128, 0, s>>>(w_in, e->w_in3, d, JF, Kp);
  CUDA_TRY(cudaGetLastError());
  TRY(dalloc(&e->w_out3, static_cast<size_t>(e->N_out_pad) * 3 * d, true));
  split_weight_kernel<<<JF, 128, 0, s>>>(w_out, e->w_out3, JF, d, d);
  CUDA_TRY(cudaGetLastError());
  TRY(make_map(&e->m_win, e->w_in3, d, 3 * Kp, 3 * Kp, 128));
  TRY(make_map(&e->m_wout, e->w_out3, e->N_out_pad, 3 * d, 3 * d, 96));

  for (int l = 0; l < e->L; ++l) {
    LayerW& w = e->layers[l];
    const std::string p = std::string(e->dec ? "seqTransDecoder.layers." : "seqTransEncoder.layers.") + std::to_string(l) + ".";
    const float *wqkv, *wo, *w1, *w2;
    TRY(need(e, p + "self_attn.in_proj_weight", {3 * d, d}, &wqkv));
    TRY(need(e, p + "self_attn.in_proj_bias", {3 * d}, &w.bqkv));
    TRY(need(e, p + "self_attn.out_proj.weight", {d, d}, &wo));
    TRY(need(e, p + "self_attn.out_proj.bias", {d}, &w.bo));
    TRY(need(e, p + "linear1.weight", {ff, d}, &w1));
    TRY(need(e, p + "linear1.bias", {ff}, &w.b1));
    TRY(need(e, p + "linear2.weight", {d, ff}, &w2));
    TRY(need(e, p + "linear2.bias", {d}, &w.b2));
    TRY(need(e, p + "norm1.weight", {d}, &w.g1));
    TRY(need(e, p + "norm1.bias", {d}, &w.be1));
    TRY(need(e, p + "norm2.weight", {d}, &w.g2));
    TRY(need(e, p + "norm2.bias", {d}, &w.be2));
    const int kw = e->kw;   // 2: weights repeated along K for [hi | lo] activations
    TRY(to_f16_k(wqkv, &w.wqkv, 3 * d, d, kw, s));
    TRY(to_f16_k(wo, &w.wo, d, d, kw, s));
    TRY(to_f16_k(w1, &w.w1, ff, d, kw, s));
    TRY(to_f16_k(w2, &w.w2, d, ff, kw, s));
    TRY(make_map(&w.m_wqkv, w.wqkv, 3 * d, kw * d, kw * d, 128));
    TRY(make_map(&w.m_wqkv_64, w.wqkv, 3 * d, kw * d, kw * d, 64));
    TRY(make_map(&w.m_wo, w.wo, d, kw * d, kw * d, 128));
    TRY(make_map(&w.m_w1, w.w1, ff, kw * d, kw * d, 128));
    TRY(make_map(&w.m_w2, w.w2, d, kw * ff, kw * ff, 128));
    TRY(make_map(&w.m_wo_256, w.wo, d, kw * d, kw * d, 256));
    TRY(make_map(&w.m_w2_256, w.w2, d, kw * ff, kw * ff, 256));
    if (e->dec) {
      // nn.MultiheadAttention in_proj rows: [Wq; Wk; Wv] -- query from the sequence, key/value from the text memory
      const float *wc, *bc, *woc;
      TRY(need(e, p + "multihead_attn.in_proj_weight", {3 * d, d}, &wc));
      TRY(need(e, p + "multihead_attn.in_proj_bias", {3 * d}, &bc));
      TRY(need(e, p + "multihead_attn.out_proj.weight", {d, d}, &woc));
      TRY(need(e, p + "multihead_attn.out_proj.bias", {d}, &w.bo_c));
      TRY(need(e, p + "norm3.weight", {d}, &w.g3));
      TRY(need(e, p + "norm3.bias", {d}, &w.be3));
      w.bq_c = bc;
      TRY(to_f16_k(wc, &w.wq_c, d, d, kw, s));
      if (l == 0) {
        TRY(dalloc(&e->wkv_all, static_cast<size_t>(e->L) * 2 * d * d));
        TRY(dalloc(&e->bkv_all, static_cast<size_t>(e->L) * 2 * d));
        TRY(make_map(&e->m_wkv_all, e->wkv_all, static_cast<uint64_t>(e->L) * 2 * d, d, d, 128));
      }
      f32_to_f16_kernel<<<512, 256, 0, s>>>(wc + static_cast<size_t>(d) * d, e->wkv_all + static_cast<size_t>(l) * 2 * d * d,
                                            static_cast<size_t>(2) * d * d);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaMemcpyAsync(e->bkv_all + static_cast<size_t>(l) * 2 * d, bc + d, sizeof(float) * 2 * d, cudaMemcpyDeviceToDevice, s));
      TRY(to_f16_k(woc, &w.wo_c, d, d, kw, s));
      TRY(make_map(&w.m_wq_c, w.wq_c, d, kw * d, kw * d, 128));
      TRY(make_map(&w.m_wo_c_256, w.wo_c, d, kw * d, kw * d, 256));
    }
  }
  // timestep-embedding MLP for every model timestep: temb[t] = W2 silu(W1 pe[t] + b1) + b2
  const int R = e->cfg.temb_rows;
  TRY(dalloc(&e->temb_hidden, static_cast<size_t>(R) * d));
  TRY(dalloc(&e->temb_table, static_cast<size_t>(R) * d));
  const size_t warps = static_cast<size_t>(R) * d;
  const int blocks = static_cast<int>((warps * 32 + 255) / 256);
  small_linear_kernel<1><<<blocks, 256, 0, s>>>(e->pe, t0w, t0b, e->temb_hidden, R, d, d, d);
  CUDA_TRY(cudaGetLastError());
  small_linear_kernel<0><<<blocks, 256, 0, s>>>(e->temb_hidden, t2w, t2b, e->temb_table, R, d, d, d);
  CUDA_TRY(cudaGetLastError());
  TRY(finalize_target(e, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  e->finalized = true;
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ schedule
extern "C" int b200mdm_set_schedule(b200mdm_engine* e, int32_t n_steps, const float* rows_host,
                                    const int32_t* timestep_map_host) {
  if (!e || n_steps <= 0 || !rows_host || !timestep_map_host) return fail(B200MDM_EINVAL, "bad argument");
  for (int i = 0; i < n_steps; ++i)
    if (timestep_map_host[i] < 0 || timestep_map_host[i] >= e->cfg.temb_rows)
      return fail(B200MDM_EINVAL, "timestep_map[%d] = %d outside the pre-embedded range [0, %d)", i, timestep_map_host[i],
                  e->cfg.temb_rows);
  CUDA_TRY(cudaDeviceSynchronize());  // a loop still in flight may be reading the old tables
  if (n_steps > e->sched_cap) {
    // the captured step graphs hold these pointers as kernel parameters: moving the tables invalidates every graph
    drop_all_graphs(e);
    dfree(e->sched);
    dfree(e->tmap);
    const int cap = n_steps > 1000 ? n_steps : 1000;
    TRY(dalloc(&e->sched, static_cast<size_t>(cap) * SCHED_STRIDE));
    TRY(dalloc(&e->tmap, cap));
    e->sched_cap = cap;
  }
  e->n_steps = n_steps;
  CUDA_TRY(cudaMemcpy(e->sched, rows_host, static_cast<size_t>(n_steps) * SCHED_STRIDE * sizeof(float), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(e->tmap, timestep_map_host, static_cast<size_t>(n_steps) * sizeof(int), cudaMemcpyHostToDevice));
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ cond / workspace
static void attach_l2_window(b200mdm_engine* e, cudaStream_t stream = nullptr);
static bool fused_qkv_enabled(int S);

static int build_workspace(b200mdm_engine* e, int B, int T, int halves, cudaStream_t s) {
  const int d = e->d, S = T + e->s_off, Bp = halves * B;
  const size_t M = static_cast<size_t>(Bp) * S, MB = static_cast<size_t>(B) * S;
  TRY(dalloc(&e->xin16, MB * 3 * e->Kp_in, true));
  const int kw = e->kw;
  TRY(dalloc(&e->hres, M * d * 2, true));   // residual stream, fp16 [hi | lo]
  const bool need_qkv = e->dec || !fused_qkv_enabled(S);   // the encoder's fused QKV + attention kernel never materialises qkv
  if (need_qkv) TRY(dalloc(&e->qkv16, M * 3 * d));
  TRY(dalloc(&e->att16, M * d * kw));
  TRY(dalloc(&e->ffn16, M * e->ff * kw));
  TRY(dalloc(&e->g16, static_cast<size_t>(B) * T * 3 * d));           // frame rows only
  TRY(dalloc(&e->tok0, static_cast<size_t>(Bp) * d));
  TRY(dalloc(&e->condproj, static_cast<size_t>(Bp) * d, true));
  TRY(dalloc(&e->proj, static_cast<size_t>(B) * d, true));
  TRY(dalloc(&e->scale, B, true));
  TRY(dalloc(&e->x_work, static_cast<size_t>(B) * e->JF * T));
  TRY(dalloc(&e->kvlen, Bp));
  TRY(dalloc(&e->tvec, B, true));
  TRY(dalloc(&e->action, B, true));
  if (e->dec) {
    TRY(dalloc(&e->qc16, M * d));
    TRY(make_map_t(&e->m_qc_st, e->qc16, 2, M, d, d, 32));
    e->Mt = 0;              // the text-memory buffers are sized by the packed batch: b200mdm_set_cond_dec rebuilds them
    e->prefix_set = false;  // xin16 was reallocated
  }
  e->B = B; e->T = T; e->S = S; e->halves = halves; e->Bp = Bp;
  e->M = static_cast<int>(M); e->MB = static_cast<int>(MB);
  attach_l2_window(e);
  TRY(make_map(&e->m_xin, e->xin16, MB, 3 * e->Kp_in, 3 * e->Kp_in, GEMM_BLOCK_M));
  // GEMM A operand = the hi half of the residual stream (kw = 2, trans_dec: both halves, K = 2d against [W | W])
  TRY(make_map(&e->m_h16, e->hres, M, kw * d, 2 * d, GEMM_BLOCK_M));
  TRY(make_map(&e->m_att, e->att16, M, kw * d, kw * d, GEMM_BLOCK_M));
  TRY(make_map(&e->m_ffn, e->ffn16, M, kw * e->ff, kw * e->ff, GEMM_BLOCK_M));
  TRY(make_map(&e->m_g16, e->g16, static_cast<size_t>(B) * T, 3 * d, 3 * d, GEMM_BLOCK_M));
  if (need_qkv) TRY(make_map_t(&e->m_qkv_st, e->qkv16, 2, M, 3 * d, 3 * d, 32));
  TRY(make_map_t(&e->m_ffn_st, e->ffn16, 2, M, kw * e->ff, kw * e->ff, 32));
  TRY(make_map_res(&e->m_res, e->hres, M, d));
  if (need_qkv) {
    AttnMaps am;
    TRY(make_attn_maps(&am, e->qkv16, e->att16, Bp, S, d, kw));
    e->m_att_q = am.q; e->m_att_kv = am.kv; e->m_att_o = am.o;
  } else {
    TRY(make_map_3d(&e->m_att_o, e->att16, Bp, S, kw * d, kw * d, 32));   // output slabs of the fused kernel
  }
  TRY(make_map_res(&e->m_res_c, e->hres, MB, d));
  TRY(make_map_res(&e->m_res_u, e->hres + (halves == 2 ? MB * d * 2 : 0), MB, d));
  TRY(dalloc(&e->pe_bias, static_cast<size_t>(S) * d));
  pe_bias_kernel<<<S, 128, 0, s>>>(e->pe_bias, e->pe, e->b_in, S, d);   // on the caller's stream: ordered before any forward
  CUDA_TRY(cudaGetLastError());
  TRY(dalloc(&e->eps_buf, static_cast<size_t>(B) * e->JF * T));
  // fused QKV + attention (qkv_attn.cuh): per-sample 3-D view of the stream's hi half (A tiles of 128 tokens that stop
  // at the sample's last token) and of att16 (128-row output tiles clipped the same way)
  TRY(make_map_3d(&e->m_h3, e->hres, Bp, S, d, 2 * d, 128));
  return B200MDM_OK;
}

// Keep the residual stream resident in the L2 (126 MB): it is read and rewritten by every residual+LayerNorm GEMM, and
// between two of them ~230 MB of other activations stream through.  The window is attached to the engine stream, so
// every kernel captured into the step graph inherits it.  Best effort: failures are ignored.
static void attach_l2_window(b200mdm_engine* e, cudaStream_t stream) {
  cudaDeviceProp prop;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaGetDeviceProperties(&prop, dev) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
    const size_t want = static_cast<size_t>(e->M) * e->d * 2 * sizeof(__half);
    const size_t carve = want < static_cast<size_t>(prop.persistingL2CacheMaxSize) ? want : static_cast<size_t>(prop.persistingL2CacheMaxSize);
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    attr.accessPolicyWindow.base_ptr = e->hres;
    attr.accessPolicyWindow.num_bytes = want < static_cast<size_t>(prop.accessPolicyMaxWindowSize) ? want : static_cast<size_t>(prop.accessPolicyMaxWindowSize);
    attr.accessPolicyWindow.hitRatio = want <= carve ? 1.0f : static_cast<float>(carve) / static_cast<float>(want);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    cudaStreamSetAttribute(stream ? stream : e->work, cudaStreamAttributeAccessPolicyWindow, &attr);
    cudaGetLastError();
  }
}

// Make the workspace for (B, T, halves) the current one: the one in use if it matches, else a parked one, else a new
// one (the least recently used of more than `MAX_PARKED` parked workspaces is freed).
static int select_workspace(b200mdm_engine* e, int B, int T, int halves, cudaStream_t s) {
  constexpr size_t MAX_PARKED = 3;
  Workspace* cur = static_cast<Workspace*>(e);
  e->last_use = ++e->use_clock;
  if (cur->B == B && cur->T == T && cur->halves == halves) return B200MDM_OK;
  if (cur->B > 0) {
    e->pool.push_back(*cur);
    *cur = Workspace();
  }
  for (size_t i = 0; i < e->pool.size(); ++i) {
    if (e->pool[i].B == B && e->pool[i].T == T && e->pool[i].halves == halves) {
      *cur = e->pool[i];
      e->pool.erase(e->pool.begin() + i);
      cur->last_use = e->use_clock;
      cur->cond_set = false;      // the caller is about to set the conditioning of this loop
      cur->prefix_set = false;
      attach_l2_window(e);
      return B200MDM_OK;
    }
  }
  while (e->pool.size() > MAX_PARKED) {
    size_t lru = 0;
    for (size_t i = 1; i < e->pool.size(); ++i)
      if (e->pool[i].last_use < e->pool[lru].last_use) lru = i;
    CUDA_TRY(cudaDeviceSynchronize());   // a loop on that workspace may still be running
    free_workspace(&e->pool[lru]);
    e->pool.erase(e->pool.begin() + lru);
  }
  int r = build_workspace(e, B, T, halves, s);
  if (r != B200MDM_OK) free_workspace(cur);
  cur->last_use = e->use_clock;
  return r;
}


// ---- target-location conditioning (model/mdm.py:197-199; encoders in target_embed.cuh)
static int launch_tgt_linear(b200mdm_engine* e, const TgtLinear& p, int groups, int max_rows, cudaStream_t s) {
  tgt_linear_kernel<<<dim3((p.N + TGT_BN - 1) / TGT_BN, (max_rows + TGT_BM - 1) / TGT_BM, groups), TGT_THREADS, 0, s>>>(p);
  CUDA_TRY(cudaGetLastError());
  e->launches++;
  return B200MDM_OK;
}

extern "C" int b200mdm_set_target(b200mdm_engine* e, int32_t batch, const float* target_cond_dev, const uint8_t* valid_host,
                                  void* stream) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  if (e->cfg.target_encoder == B200MDM_TARGET_NONE)
    return fail(B200MDM_EINVAL, "this engine has no target encoder (created with target_encoder = 0)");
  e->tgt_pending = false;
  if (!target_cond_dev) return B200MDM_OK;   // no target / target_uncond: the conditioning rows stay exactly as without
  if (!e->finalized) return fail(B200MDM_ESTATE, "weights not finalised");
  if (batch <= 0 || !valid_host) return fail(B200MDM_EINVAL, "bad batch / null validity mask");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int d = e->d, n = e->cfg.n_goal_rows, B = batch, type = e->cfg.target_encoder;
  const int hcols = type == B200MDM_TARGET_MULTI ? n * d : d;   // per-sample width of the hidden buffers
  if (B > e->tgt_cap) {
    CUDA_TRY(cudaDeviceSynchronize());   // a set_cond* of an earlier loop may still read the old buffer
    dfree(e->tgt_out); dfree(e->tgt_ha); dfree(e->tgt_hb); dfree(e->tgt_x0); dfree(e->tgt_idx);
    e->tgt_cap = 0;
    TRY(dalloc(&e->tgt_out, static_cast<size_t>(B) * d));
    TRY(dalloc(&e->tgt_ha, static_cast<size_t>(B) * hcols));
    TRY(dalloc(&e->tgt_hb, static_cast<size_t>(B) * hcols));
    TRY(dalloc(&e->tgt_x0, static_cast<size_t>(B) * 4 * n));
    TRY(dalloc(&e->tgt_idx, static_cast<size_t>(n) + 2 * static_cast<size_t>(n) * B));
    e->tgt_cap = B;
  }
  // host staging: per-row sample lists (multi encoder) and the validity mask as ints
  std::vector<int>& h = e->h_tgt;
  h.assign(static_cast<size_t>(n) + 2 * static_cast<size_t>(n) * B, 0);
  int* counts = h.data();
  int* lists = counts + n;
  int* valid = lists + static_cast<size_t>(n) * B;
  for (int b = 0; b < B; ++b)
    for (int j = 0; j < n; ++j)
      if (valid_host[static_cast<size_t>(b) * n + j]) {
        valid[static_cast<size_t>(b) * n + j] = 1;
        lists[static_cast<size_t>(j) * B + counts[j]++] = b;
      }
  CUDA_TRY(cudaMemcpyAsync(e->tgt_idx, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  const int* d_counts = e->tgt_idx;
  const int* d_lists = e->tgt_idx + n;
  const int* d_valid = e->tgt_idx + n + static_cast<size_t>(n) * B;
  const std::vector<TgtStage> st = target_stages(e->cfg);
  if (type == B200MDM_TARGET_MULTI) {
    // e_j = L2_j(SiLU(L1_j(target[b, j]))) for the samples whose row j is valid: one group per row, its own sample list
    int max_rows = 0;
    for (int j = 0; j < n; ++j) max_rows = counts[j] > max_rows ? counts[j] : max_rows;
    if (max_rows > 0) {
      for (int k = 0; k < 2; ++k) {
        TgtLinear p{};
        p.x = k == 0 ? target_cond_dev : e->tgt_ha;
        p.x_gs = k == 0 ? 3 : static_cast<long long>(B) * d;
        p.ldx = k == 0 ? 3 * n : d;
        p.w = e->tgt_w[k]; p.w_gs = static_cast<long long>(st[k].N) * st[k].K;
        p.bias = e->tgt_b[k]; p.b_gs = st[k].N;
        p.y = k == 0 ? e->tgt_ha : e->tgt_hb; p.y_gs = static_cast<long long>(B) * d; p.ldy = d;
        p.rows = d_lists; p.counts = d_counts; p.rows_gs = B;
        p.R = B; p.N = st[k].N; p.K = st[k].K; p.silu_in = k;
        TRY(launch_tgt_linear(e, p, n, max_rows, s));
      }
    }
    tgt_weighted_sum_kernel<<<B, 128, 0, s>>>(e->tgt_hb, e->tgt_wn, d_valid, e->tgt_out, B, n, d);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
  } else {
    // single: one MLP on [target | valid].view(B, 4n); split: n MLPs side by side, row j reads columns 4j..4j+3 of the
    // same input and owns output columns j*d/n .. (j+1)*d/n
    tgt_input_kernel<<<(B * n * 4 + 255) / 256, 256, 0, s>>>(target_cond_dev, d_valid, e->tgt_x0, B, n);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    const bool split = type == B200MDM_TARGET_SPLIT;
    const float* x = e->tgt_x0;
    for (size_t k = 0; k < st.size(); ++k) {
      float* y = k + 1 == st.size() ? e->tgt_out : (k % 2 == 0 ? e->tgt_ha : e->tgt_hb);
      TgtLinear p{};
      p.x = x;
      p.x_gs = split ? (k == 0 ? 4 : st[k].K) : 0;
      p.ldx = k == 0 ? 4 * n : d;
      p.w = e->tgt_w[k]; p.w_gs = static_cast<long long>(st[k].N) * st[k].K;
      p.bias = e->tgt_b[k]; p.b_gs = st[k].N;
      p.y = y; p.y_gs = split ? st[k].N : 0; p.ldy = d;
      p.R = B; p.N = st[k].N; p.K = st[k].K; p.silu_in = k > 0 ? 1 : 0;
      TRY(launch_tgt_linear(e, p, st[k].groups, B, s));
      x = y;
    }
  }
  e->tgt_batch = B;
  e->tgt_pending = true;
  return B200MDM_OK;
}

// The target embedding b200mdm_set_target left for this set_cond* call (nullptr: none); it is consumed either way.
static int take_target(b200mdm_engine* e, int batch, const float** tgt) {
  *tgt = nullptr;
  if (!e->tgt_pending) return B200MDM_OK;
  e->tgt_pending = false;
  if (e->tgt_batch != batch)
    return fail(B200MDM_EINVAL, "b200mdm_set_target was called for batch %d, the conditioning is for batch %d", e->tgt_batch, batch);
  *tgt = e->tgt_out;
  return B200MDM_OK;
}

extern "C" int b200mdm_set_cond(b200mdm_engine* e, int32_t batch, int32_t nframes, const float* cond_embed_dev,
                                const int64_t* lengths_host, const float* scale_dev, int32_t force_uncond,
                                const int64_t* action_host, void* stream) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  if (e->dec) return fail(B200MDM_EINVAL, "trans_dec engines take their conditioning through b200mdm_set_cond_dec");
  const float* tgt = nullptr;
  TRY(take_target(e, batch, &tgt));
  if (!e->finalized) return fail(B200MDM_ESTATE, "weights not finalised");
  if (batch <= 0 || nframes <= 0) return fail(B200MDM_EINVAL, "bad batch / nframes");
  if (nframes + 1 > e->cfg.pos_embed_max_len) return fail(B200MDM_EINVAL, "sequence longer than the positional table");
  if (nframes + 1 > ATC_MAX_KEYS)
    return fail(B200MDM_ENOTIMPL, "sequences of more than %d tokens (the attention kernels keep all keys of a sample on chip; "
                "every dataset of the reference stops at 196 frames)", ATC_MAX_KEYS);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int halves = scale_dev ? 2 : 1;
  if (e->cfg.cond_mode == B200MDM_COND_TEXT && !cond_embed_dev && !(halves == 1 && force_uncond))
    return fail(B200MDM_EINVAL, "text-conditioned model needs y['text_embed']");
  if (e->cfg.cond_mode == B200MDM_COND_ACTION && !action_host && !(halves == 1 && force_uncond))
    return fail(B200MDM_EINVAL, "action-conditioned model needs y['action']");
  if (halves == 2 && e->cfg.cond_mode == B200MDM_COND_NONE)
    return fail(B200MDM_EINVAL, "classifier-free guidance needs a conditioned model (sampler_util.py:29)");
  TRY(select_workspace(e, batch, nframes, halves, s));
  const int d = e->d, B = batch, S = nframes + 1;
  // key mask -> valid-key counts (model/mdm.py:241-247; lengths_to_mask, data_loaders/tensors.py:3-6)
  // (host staging lives in the engine until the next call, so the asynchronous copies need no stream synchronisation)
  std::vector<int>& kv = e->h_kv;
  kv.assign(e->Bp, S);
  if (e->cfg.mask_frames && lengths_host && nframes > 1) {
    for (int b = 0; b < e->Bp; ++b) {
      long long len = lengths_host[b % B];
      if (len < 0) len = 0;
      if (len > nframes) len = nframes;
      kv[b] = static_cast<int>(len) + 1;
    }
  }
  CUDA_TRY(cudaMemcpyAsync(e->kvlen, kv.data(), kv.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  if (scale_dev) CUDA_TRY(cudaMemcpyAsync(e->scale, scale_dev, B * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (e->cfg.cond_mode == B200MDM_COND_ACTION && action_host) {
    std::vector<int>& a = e->h_action;
    a.assign(B, 0);
    for (int b = 0; b < B; ++b) {
      if (action_host[b] < 0 || action_host[b] >= e->cfg.num_actions) return fail(B200MDM_EINVAL, "action index out of range");
      a[b] = static_cast<int>(action_host[b]);
    }
    CUDA_TRY(cudaMemcpyAsync(e->action, a.data(), B * sizeof(int), cudaMemcpyHostToDevice, s));
  }
  if (e->cfg.cond_mode == B200MDM_COND_TEXT && cond_embed_dev) {
    const size_t warps = static_cast<size_t>(B) * d;
    small_linear_kernel<0><<<static_cast<int>((warps * 32 + 255) / 256), 256, 0, s>>>(cond_embed_dev, e->w_txt, e->b_txt, e->proj, B,
                                                                                       d, e->cfg.cond_dim, e->cfg.cond_dim);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
  }
  condproj_fill_kernel<<<e->Bp, 128, 0, s>>>(e->condproj, e->proj, e->b_txt, e->act_emb, e->action, B, d, e->Bp,
                                             (halves == 1 && force_uncond) ? 1 : 0, e->cfg.cond_mode, tgt);
  CUDA_TRY(cudaGetLastError());
  e->launches++;
  e->cond_set = true;
  return B200MDM_OK;
}

// ---- trans_dec (DiP) conditioning: BERT token features + padding mask as the cross-attention memory, prefix frames
extern "C" int b200mdm_set_cond_dec(b200mdm_engine* e, int32_t batch, int32_t nframes, const float* enc_text_dev,
                                    const uint8_t* text_mask_host, int32_t n_tokens, const int64_t* lengths_host,
                                    const float* scale_dev, int32_t force_uncond, void* stream) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  if (!e->dec) return fail(B200MDM_EINVAL, "b200mdm_set_cond_dec is for trans_dec engines");
  const float* tgt = nullptr;
  TRY(take_target(e, batch, &tgt));
  if (!e->finalized) return fail(B200MDM_ESTATE, "weights not finalised");
  if (batch <= 0 || nframes <= 0 || n_tokens <= 0 || n_tokens > 64) return fail(B200MDM_EINVAL, "bad batch / nframes / n_tokens (1..64)");
  if (nframes + e->ctx > e->cfg.pos_embed_max_len) return fail(B200MDM_EINVAL, "sequence longer than the positional table");
  if (nframes + e->ctx > ATC_MAX_KEYS) return fail(B200MDM_ENOTIMPL, "sequences of more than %d tokens", ATC_MAX_KEYS);
  if (!enc_text_dev || !text_mask_host) return fail(B200MDM_EINVAL, "DiP needs y['text_embed'] = (tokens, mask)");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int halves = scale_dev ? 2 : 1;
  TRY(select_workspace(e, batch, nframes, halves, s));
  const int d = e->d, B = batch, S = e->S, Bp = e->Bp, Mt = n_tokens, C = e->cfg.cond_dim;
  if (Mt != e->Mt) {
    CUDA_TRY(cudaDeviceSynchronize());
    drop_graph(e);
    dfree(e->encperm); dfree(e->memtok); dfree(e->memproj); dfree(e->mem16); dfree(e->kvc16); dfree(e->memmask);
    TRY(dalloc(&e->encperm, static_cast<size_t>(B) * Mt * C));
    TRY(dalloc(&e->memtok, static_cast<size_t>(B) * Mt * d));
    TRY(dalloc(&e->memproj, static_cast<size_t>(Bp) * Mt * d));
    TRY(dalloc(&e->mem16, static_cast<size_t>(Bp) * Mt * 2 * d));   // [hi | lo]
    TRY(dalloc(&e->kvc16, static_cast<size_t>(Bp) * Mt * 2 * d * e->L));      // [Bp*Mt, L * (k | v)]
    TRY(dalloc(&e->memmask, static_cast<size_t>(Bp) * Mt));
    TRY(make_map(&e->m_mem, e->mem16, static_cast<uint64_t>(Bp) * Mt, 2 * d, 2 * d, GEMM_BLOCK_M));
    TRY(make_map_t(&e->m_kvc_st, e->kvc16, 2, static_cast<uint64_t>(Bp) * Mt, 2 * d * e->L, 2 * d * e->L, 32));
    e->Mt = Mt;
  }
  // key mask of the frames: the context frames are always valid (model/mdm.py:204-206), then `lengths` frames of x
  std::vector<int>& kv = e->h_kv;
  kv.assign(Bp, S);
  if (e->cfg.mask_frames && lengths_host && S > 1) {
    for (int b = 0; b < Bp; ++b) {
      long long len = lengths_host[b % B];
      if (len < 0) len = 0;
      if (len > nframes) len = nframes;
      kv[b] = static_cast<int>(len) + e->ctx;
    }
  }
  std::vector<unsigned char>& mk = e->h_mask;
  mk.assign(static_cast<size_t>(Bp) * Mt, 0);
  for (int b = 0; b < Bp; ++b)
    for (int m = 0; m < Mt; ++m) mk[static_cast<size_t>(b) * Mt + m] = text_mask_host[static_cast<size_t>(b % B) * Mt + m] ? 1 : 0;
  CUDA_TRY(cudaMemcpyAsync(e->kvlen, kv.data(), kv.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->memmask, mk.data(), mk.size(), cudaMemcpyHostToDevice, s));
  if (scale_dev) CUDA_TRY(cudaMemcpyAsync(e->scale, scale_dev, B * sizeof(float), cudaMemcpyDeviceToDevice, s));
  // text_emb = embed_text(mask_cond(enc_text)) per token (model/mdm.py:218), once per loop
  permute_mbc_kernel<<<dim3(Mt, B), 128, 0, s>>>(enc_text_dev, e->encperm, Mt, B, C);
  CUDA_TRY(cudaGetLastError());
  const size_t warps = static_cast<size_t>(B) * Mt * d;
  small_linear_kernel<0><<<static_cast<int>((warps * 32 + 255) / 256), 256, 0, s>>>(e->encperm, e->w_txt, e->b_txt, e->memtok, B * Mt, d, C, C);
  CUDA_TRY(cudaGetLastError());
  memproj_fill_kernel<<<dim3(Mt, Bp), 128, 0, s>>>(e->memproj, e->memtok, e->b_txt, B, Mt, d, Bp, (halves == 1 && force_uncond) ? 1 : 0,
                                                   tgt);
  CUDA_TRY(cudaGetLastError());
  e->launches += 3;
  e->cond_set = true;
  return B200MDM_OK;
}

// y['prefix'] [B, J, F, context_len] (model/mdm.py:203-206): packed once per loop into the first context_len rows of
// every sequence of the embedding GEMM's A operand.
extern "C" int b200mdm_set_prefix(b200mdm_engine* e, const float* prefix_dev, void* stream) {
  if (!e || !prefix_dev) return fail(B200MDM_EINVAL, "null argument");
  if (!e->dec || e->ctx <= 0) return fail(B200MDM_EINVAL, "this engine has no prefix (context_len == 0)");
  if (!e->cond_set) return fail(B200MDM_ESTATE, "call b200mdm_set_cond_dec first (it sizes the workspace)");
  dim3 grid((e->ctx + 31) / 32, (e->JF + 31) / 32, e->B), block(32, 8);
  pack_input_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(prefix_dev, e->xin16, e->B, e->JF, e->ctx, e->S, e->Kp_in,
                                                                          3 * e->Kp_in, 0);
  CUDA_TRY(cudaGetLastError());
  e->launches++;
  e->prefix_set = true;
  return B200MDM_OK;
}

extern "C" int b200mdm_set_inpaint(b200mdm_engine* e, const uint8_t* mask_dev, const float* motion_dev) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  if ((mask_dev == nullptr) != (motion_dev == nullptr)) return fail(B200MDM_EINVAL, "inpainting needs both mask and motion");
  e->inpaint_mask = mask_dev;
  e->inpaint_motion = motion_dev;
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ forward
struct StepArgs {
  int mode = B200MDM_MODE_X0;
  const float* x_in = nullptr;    // [B, JF, T] input to the denoiser (x_t)
  const float* noise = nullptr;   // explicit eps (single step); nullptr => tape from the device step state
  int const_noise = 0;
  int clip = 0;
  float* x_out = nullptr;
  float* pred = nullptr;
  bool explicit_t = false;        // use e->tvec instead of timestep_map[state.cur]
  bool philox = false;            // eps of this step is generated into e->eps_buf by the first kernel of the step
};

// Enqueue one denoiser forward (+ fused sampler step) on stream s.  Returns the number of kernels launched.
static int enqueue_forward(b200mdm_engine* e, const StepArgs& a, cudaStream_t s, int* n_kernels) {
  const int d = e->d, ff = e->ff, B = e->B, T = e->T, S = e->S, JF = e->JF, Kp = e->Kp_in;
  int nk = 0;
  PdlScope pdl_scope;
  if (a.philox) {
    const long long quads = (static_cast<long long>(JF) * T + 3) / 4 * B;
    const int blocks = static_cast<int>(quads / 256 + 1 < 1184 ? quads / 256 + 1 : 1184);
    CUDA_TRY(launch_k(philox_normal_kernel, dim3(blocks), dim3(256), 0, s, e->eps_buf, B, static_cast<long long>(JF) * T,
                      0ull, 0ll, 0u, e->state));
    ++nk;
  }
  {
    dim3 grid((T + 31) / 32, (JF + 31) / 32, B), block(32, 8);
    CUDA_TRY(launch_k(pack_input_kernel, grid, block, 0, s, a.x_in, e->xin16, B, JF, T, S, Kp, 3 * Kp, e->s_off));
    ++nk;
  }
  {
    EpiEmbed::Params p;
    p.res_c = e->m_res_c; p.res_u = e->m_res_u;
    p.pe_bias = e->pe_bias;
    p.S = S; p.d = d; p.halves = e->halves;
    TRY((launch_gemm<128, EpiEmbed>(e->m_xin, e->m_win, e->m_xin, e->MB, d, 3 * Kp, p, s, e->num_sms)));
    ++nk;
  }
  if (!e->dec) {
    CUDA_TRY(launch_k(tok0_rows_kernel, dim3(e->Bp), dim3(128), 0, s, e->hres, e->condproj, e->temb_table, e->pe,
                      a.explicit_t ? e->tvec : nullptr, e->tmap, e->state, B, S, d, e->cfg.temb_rows));
  } else {
    // cross-attention memory of this step: text tokens + timestep embedding (model/mdm.py:218-220)
    CUDA_TRY(launch_k(mem_build_kernel, dim3(e->Mt, e->Bp), dim3(128), 0, s, e->mem16, e->memproj, e->temb_table,
                      a.explicit_t ? e->tvec : nullptr, e->tmap, e->state, B, e->Mt, d, e->cfg.temb_rows));
    // ... and its key / value projections for every layer in one GEMM (N = L * 2d; hi half of the memory, K = d)
    EpiBiasF16Global::Params p{e->bkv_all};
    TRY((launch_gemm2<EpiBiasF16Global>(e->m_mem, e->m_wkv_all, e->m_kvc_st, e->Bp * e->Mt, e->L * 2 * d, d, p, s, e->num_sms)));
    ++nk;
  }
  ++nk;
  const int kw = e->kw;
  const bool wide = kw == 2;
  for (int l = 0; l < e->L; ++l) {
    const LayerW& w = e->layers[l];
    if (B200_SKIP(1)) {
      ++nk;
    } else if (!wide && fused_qkv_enabled(S)) {
      // QKV projection + attention in one kernel: the [M, 1536] qkv tensor never exists
      TRY(launch_qkv_attention(e->m_h3, w.m_wqkv, w.m_wqkv_64, e->m_att_o, w.bqkv, e->kvlen, e->Bp, S, s, e->num_sms));
      --nk;
    } else {
      {
        // trans_dec keeps [hi | lo] activations only where the precision study needs them (self-attention output,
        // FFN-up input, FFN-down input: oracle emulation 6.2e-4 vs 5.1e-4 with every site split, tolerance 1e-3); the
        // projections below read the hi half alone: K = d against the first d columns of [W | W]
        TRY((launch_gemm2_bias<false>(e->m_h16, w.m_wqkv, e->m_qkv_st, e->M, 3 * d, d, w.bqkv, s, e->num_sms)));
      }
      AttnMaps am{e->m_att_q, e->m_att_kv, e->m_att_o};
      TRY(launch_attention_tc(am, e->kvlen, e->Bp, S, d, e->H, s, wide));
    }
    if (!B200_SKIP(2)) TRY(launch_gemm_resid_ln(e->m_att, w.m_wo_256, e->m_res, e->M, kw * d, w.bo, w.g1, w.be1, s, e->num_sms));
    if (e->dec) {
      // cross-attention block of nn.TransformerDecoderLayer: q from the sequence, k/v from the text memory
      TRY((launch_gemm2_bias<false>(e->m_h16, w.m_wq_c, e->m_qc_st, e->M, d, d, w.bq_c, s, e->num_sms)));
      {
        const float sl2 = 1.4426950408889634f / sqrtf(128.0f);
        const dim3 cg(e->H, e->Bp), cb(128);
        const __half* kvl = e->kvc16 + static_cast<size_t>(l) * 2 * d;      // this layer's k | v columns
        const int ldkv = e->L * 2 * d;
        if (e->Mt <= 16)
          CUDA_TRY(launch_k(cross_attention_kernel<2>, cg, cb, 0, s, e->qc16, kvl, e->memmask, e->att16, S, e->Mt, d, ldkv, sl2));
        else if (e->Mt <= 32)
          CUDA_TRY(launch_k(cross_attention_kernel<4>, cg, cb, 0, s, e->qc16, kvl, e->memmask, e->att16, S, e->Mt, d, ldkv, sl2));
        else
          CUDA_TRY(launch_k(cross_attention_kernel<8>, cg, cb, 0, s, e->qc16, kvl, e->memmask, e->att16, S, e->Mt, d, ldkv, sl2));
      }
      TRY(launch_gemm_resid_ln(e->m_att, w.m_wo_c_256, e->m_res, e->M, d, w.bo_c, w.g2, w.be2, s, e->num_sms));   // cross-attention output: hi half
      nk += 3;
    }
    if (wide) {
      EpiBiasF16Wide<true>::Params p{w.b1, ff};
      TRY((launch_gemm2<EpiBiasF16Wide<true>>(e->m_h16, w.m_w1, e->m_ffn_st, e->M, ff, kw * d, p, s, e->num_sms)));
    } else if (!B200_SKIP(4)) {
      // K = d: each CTA's half of a W1 tile stays in shared memory for the whole launch (gemm2w.cuh)
      TRY((launch_gemm2_bias<true>(e->m_h16, w.m_w1, e->m_ffn_st, e->M, ff, d, w.b1, s, e->num_sms)));
    }
    if (!B200_SKIP(8)) TRY(launch_gemm_resid_ln(e->m_ffn, w.m_w2_256, e->m_res, e->M, kw * ff, w.b2, e->dec ? w.g3 : w.g2,
                             e->dec ? w.be3 : w.be2, s, e->num_sms));
    nk += 5;
  }
  CUDA_TRY(launch_k(blend_split_kernel, dim3((B * T + 7) / 8), dim3(256), 0, s, e->hres, e->g16, e->scale, B, S, T, e->s_off, d,
                    e->halves));
  ++nk;
  {
    EpiOutStep::Params p;
    p.bias = e->b_out;
    p.x_t = a.x_in;
    p.noise = a.noise;
    p.x_out = a.x_out;
    p.pred_xstart = a.pred;
    p.inpaint_mask = e->inpaint_mask;
    p.inpaint_motion = e->inpaint_motion;
    p.sched = e->sched;
    p.state = e->state;
    p.noise_batch_stride = a.const_noise ? 0 : static_cast<long long>(JF) * T;
    p.B = B; p.S = T; p.T = T; p.J = JF; p.mode = a.mode;      // g16 rows are frames: row = b*T + t
    p.s_off = 0;
    p.clip_denoised = a.clip;
    TRY((launch_gemm<96, EpiOutStep>(e->m_g16, e->m_wout, e->m_g16, B * T, e->N_out_pad, 3 * d, p, s, e->num_sms)));
    ++nk;
  }
  *n_kernels = nk;
  return B200MDM_OK;
}

static int check_ready(b200mdm_engine* e, bool need_sched) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  if (!e->finalized) return fail(B200MDM_ESTATE, "weights not finalised");
  if (!e->cond_set) return fail(B200MDM_ESTATE, "b200mdm_set_cond has not been called");
  if (e->dec && e->ctx > 0 && !e->prefix_set) return fail(B200MDM_ESTATE, "b200mdm_set_prefix has not been called (y['prefix'])");
  if (need_sched && e->n_steps <= 0) return fail(B200MDM_ESTATE, "b200mdm_set_schedule has not been called");
  return B200MDM_OK;
}

extern "C" int b200mdm_denoise(b200mdm_engine* e, const float* x_dev, const int32_t* timesteps_host, float* out_dev,
                               void* stream) {
  TRY(check_ready(e, false));
  if (!x_dev || !timesteps_host || !out_dev) return fail(B200MDM_EINVAL, "null tensor");
  for (int b = 0; b < e->B; ++b)
    if (timesteps_host[b] < 0 || timesteps_host[b] >= e->cfg.temb_rows)
      return fail(B200MDM_EINVAL, "timestep %d outside the pre-embedded range [0, %d)", timesteps_host[b], e->cfg.temb_rows);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemcpyAsync(e->tvec, timesteps_host, e->B * sizeof(int), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // timesteps_host is caller memory
  StepArgs a;
  a.mode = B200MDM_MODE_X0;
  a.x_in = x_dev;
  a.x_out = out_dev;
  a.explicit_t = true;
  int nk = 0;
  TRY(enqueue_forward(e, a, s, &nk));
  e->launches += nk;
  return B200MDM_OK;
}

extern "C" int b200mdm_sample_step(b200mdm_engine* e, int32_t mode, int32_t index, const float* x_t_dev,
                                   const float* noise_dev, int32_t flags, float* x_out_dev,
                                   float* pred_xstart_dev, void* stream) {
  TRY(check_ready(e, true));
  if (mode != B200MDM_MODE_DDPM && mode != B200MDM_MODE_DDIM) return fail(B200MDM_EINVAL, "bad mode");
  if (index < 0 || index >= e->n_steps) return fail(B200MDM_EINVAL, "schedule index out of range");
  if (!x_t_dev || !noise_dev || !x_out_dev) return fail(B200MDM_EINVAL, "null tensor");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  step_set_kernel<<<1, 1, 0, s>>>(e->state, 0, index, nullptr, 0, e->noise_seed, e->noise_sample_base);
  CUDA_TRY(cudaGetLastError());
  StepArgs a;
  a.mode = mode;
  a.x_in = x_t_dev;
  a.noise = noise_dev;
  a.const_noise = flags & B200MDM_FLAG_CONST_NOISE;
  a.clip = (flags & B200MDM_FLAG_CLIP_DENOISED) ? 1 : 0;
  a.x_out = x_out_dev;
  a.pred = pred_xstart_dev;
  int nk = 0;
  TRY(enqueue_forward(e, a, s, &nk));
  e->launches += nk + 1;
  return B200MDM_OK;
}

// Schedule indices first_index, first_index-1, ... (n_run of them) on the engine's working buffer.  x_in_dev == NULL
// continues from the state the previous call left there; x_out_dev == NULL leaves the result there.
extern "C" int b200mdm_sample_loop_range(b200mdm_engine* e, int32_t mode, int32_t first_index, int32_t n_run,
                                         const float* x_in_dev, float* x_out_dev, const float* noise_tape_dev,
                                         int64_t noise_step_stride, int32_t flags, int32_t use_graph, void* stream) {
  TRY(check_ready(e, true));
  if (mode != B200MDM_MODE_DDPM && mode != B200MDM_MODE_DDIM) return fail(B200MDM_EINVAL, "bad mode");
  if (n_run <= 0 || first_index >= e->n_steps || first_index - n_run + 1 < 0) return fail(B200MDM_EINVAL, "bad step range");
  const bool philox = (flags & B200MDM_FLAG_PHILOX_NOISE) != 0;
  if (!philox && !noise_tape_dev) return fail(B200MDM_EINVAL, "null noise tape (or pass B200MDM_FLAG_PHILOX_NOISE)");
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  const size_t x_bytes = static_cast<size_t>(e->B) * e->JF * e->T * sizeof(float);
  // The loop runs in place on an engine-owned buffer (fixed address => the captured step graph never changes);
  // every element is read and written by the same thread of the fused output epilogue.
  StepArgs a;
  a.mode = mode;
  a.x_in = e->x_work;
  a.x_out = e->x_work;
  a.noise = philox ? e->eps_buf : nullptr;
  a.philox = philox;
  a.const_noise = flags & B200MDM_FLAG_CONST_NOISE;
  a.clip = (flags & B200MDM_FLAG_CLIP_DENOISED) ? 1 : 0;

  // The graph path runs on the engine's own stream (the caller's may be the legacy default stream, which cannot be
  // captured), ordered after / before the caller's stream with events.
  cudaStream_t s = use_graph ? e->work : user;
  if (!use_graph) attach_l2_window(e, user);   // plain launches: the residual-stream window goes on the caller's stream
  if (use_graph) {
    GraphKey key;
    key.mode = mode; key.B = e->B; key.T = e->T; key.flags = flags;
    key.imask = e->inpaint_mask; key.imotion = e->inpaint_motion;
    if (!e->graph_exec || !(key == e->graph_key)) {
      drop_graph(e);
      cudaGraph_t graph = nullptr;
      CUDA_TRY(cudaStreamBeginCapture(e->work, cudaStreamCaptureModeThreadLocal));
      int nk = 0;
      int r = enqueue_forward(e, a, e->work, &nk);
      if (r == B200MDM_OK) {
        PdlScope pdl_scope;
        if (launch_k(step_advance_kernel, dim3(1), dim3(1), 0, e->work, e->state) != cudaSuccess)
          r = fail(B200MDM_ECUDA, "step_advance launch failed during capture");
      }
      cudaError_t ce = cudaStreamEndCapture(e->work, &graph);
      if (r != B200MDM_OK) {
        if (graph) cudaGraphDestroy(graph);
        return r;
      }
      if (ce != cudaSuccess) return fail(B200MDM_ECUDA, "graph capture failed: %s", cudaGetErrorString(ce));
      ce = cudaGraphInstantiate(&e->graph_exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        e->graph_exec = nullptr;
        return fail(B200MDM_ECUDA, "graph instantiate failed: %s", cudaGetErrorString(ce));
      }
      e->graph_key = key;
      e->graph_kernels = nk + 1;
    }
    CUDA_TRY(cudaEventRecord(e->ev_in, user));
    CUDA_TRY(cudaStreamWaitEvent(e->work, e->ev_in, 0));
  }
  if (x_in_dev) CUDA_TRY(cudaMemcpyAsync(e->x_work, x_in_dev, x_bytes, cudaMemcpyDeviceToDevice, s));
  step_set_kernel<<<1, 1, 0, s>>>(e->state, 0, first_index, noise_tape_dev, noise_step_stride, e->noise_seed, e->noise_sample_base);
  CUDA_TRY(cudaGetLastError());
  e->launches += 1;
  if (use_graph) {
    for (int k = 0; k < n_run; ++k) CUDA_TRY(cudaGraphLaunch(e->graph_exec, s));
    e->launches += static_cast<long long>(n_run) * e->graph_kernels;
  } else {
    for (int k = 0; k < n_run; ++k) {
      int nk = 0;
      TRY(enqueue_forward(e, a, s, &nk));
      {
        PdlScope pdl_scope;
        CUDA_TRY(launch_k(step_advance_kernel, dim3(1), dim3(1), 0, s, e->state));
      }
      e->launches += nk + 1;
    }
  }
  if (x_out_dev) CUDA_TRY(cudaMemcpyAsync(x_out_dev, e->x_work, x_bytes, cudaMemcpyDeviceToDevice, s));
  if (use_graph) {
    CUDA_TRY(cudaEventRecord(e->ev_out, e->work));
    CUDA_TRY(cudaStreamWaitEvent(user, e->ev_out, 0));
  }
  return B200MDM_OK;
}

extern "C" int b200mdm_sample_loop(b200mdm_engine* e, int32_t mode, int32_t skip_timesteps, const float* x_T_dev,
                                   float* x_0_dev, const float* noise_tape_dev, int64_t noise_step_stride,
                                   int32_t flags, int32_t use_graph, void* stream) {
  TRY(check_ready(e, true));
  if (skip_timesteps < 0 || skip_timesteps >= e->n_steps) return fail(B200MDM_EINVAL, "bad skip_timesteps");
  if (!x_T_dev || !x_0_dev) return fail(B200MDM_EINVAL, "null tensor");
  return b200mdm_sample_loop_range(e, mode, e->n_steps - 1 - skip_timesteps, e->n_steps - skip_timesteps, x_T_dev, x_0_dev,
                                   noise_tape_dev, noise_step_stride, flags, use_graph, stream);
}

// Counter-based noise stream of the engine (Philox4x32-10 + Box-Muller, kernels.cuh): eps of schedule index i for
// global sample g depends on (seed, i, g, element) only -- not on the batch split, the GPU count or the chunking.
extern "C" int b200mdm_set_noise_stream(b200mdm_engine* e, uint64_t seed, int64_t sample_index_base) {
  if (!e) return fail(B200MDM_EINVAL, "null engine");
  e->noise_seed = seed;
  e->noise_sample_base = sample_index_base;
  return B200MDM_OK;
}
extern "C" int b200mdm_philox_normal(float* out_dev, int32_t batch, int64_t n_per_sample, uint64_t seed,
                                     int64_t sample_index_base, int32_t step_id, void* stream) {
  if (!out_dev || batch <= 0 || n_per_sample <= 0) return fail(B200MDM_EINVAL, "bad argument");
  const long long quads = (n_per_sample + 3) / 4 * batch;
  const int blocks = static_cast<int>(quads / 256 + 1 < 1184 ? quads / 256 + 1 : 1184);
  philox_normal_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(out_dev, batch, n_per_sample, seed, sample_index_base,
                                                                             static_cast<uint32_t>(step_id), nullptr);
  CUDA_TRY(cudaGetLastError());
  return B200MDM_OK;
}

extern "C" int b200mdm_q_sample(b200mdm_engine* e, float sqrt_ac, float sqrt_1mac, const float* x_start_dev,
                                const float* noise_dev, float* out_dev, int64_t n, void* stream) {
  if (!e || !noise_dev || !out_dev || n <= 0) return fail(B200MDM_EINVAL, "bad argument");
  q_sample_kernel<<<592, 256, 0, static_cast<cudaStream_t>(stream)>>>(out_dev, x_start_dev, noise_dev, sqrt_ac, sqrt_1mac,
                                                                     static_cast<size_t>(n));
  CUDA_TRY(cudaGetLastError());
  e->launches++;
  return B200MDM_OK;
}

extern "C" int64_t b200mdm_launch_count(b200mdm_engine* e, int32_t reset) {
  if (!e) return 0;
  long long v = e->launches;
  if (reset) e->launches = 0;
  return v;
}

// ------------------------------------------------------------------------------------------------ kernel tests
template <int BN>
static int test_gemm_bn(const void* a16, const void* w16, const float* bias, void* out16, int M, int N, int K, int act,
                        cudaStream_t s, int sms) {
  CUtensorMap ma, mb, mc;
  TRY(make_map(&ma, a16, M, K, K, GEMM_BLOCK_M));
  TRY(make_map(&mb, w16, N, K, K, BN));
  TRY(make_map_t(&mc, out16, 2, M, N, N, 32));
  if (act) {
    EpiBiasF16<true>::Params p{bias};
    return launch_gemm<BN, EpiBiasF16<true>>(ma, mb, mc, M, N, K, p, s, sms);
  }
  EpiBiasF16<false>::Params p{bias};
  return launch_gemm<BN, EpiBiasF16<false>>(ma, mb, mc, M, N, K, p, s, sms);
}

extern "C" int b200mdm_test_gemm_f16(const void* a16_dev, const void* w16_dev, const float* bias_dev, void* out16_dev,
                                     int32_t M, int32_t N, int32_t K, int32_t act, int32_t block_n, void* stream) {
  if (!a16_dev || !w16_dev || !bias_dev || !out16_dev || M <= 0 || N <= 0 || K <= 0 || K % 8 || N % 8)
    return fail(B200MDM_EINVAL, "bad argument (K %% 8 == 0, N %% 8 == 0 required)");
  TRY(init_kernel_attrs());
  int dev = 0, sms = 148;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (block_n == 512 || block_n == 513) {  // CTA-pair kernels, 256 x 256 pair tiles: 512 streaming, 513 W-resident
    CUtensorMap ma, mb, mc;
    TRY(make_map(&ma, a16_dev, M, K, K, GEMM_BLOCK_M));
    TRY(make_map(&mb, w16_dev, N, K, K, 128));
    TRY(make_map_t(&mc, out16_dev, 2, M, N, N, 32));
    if (block_n == 513)
      return act ? launch_gemm2w<true>(ma, mb, mc, M, N, K, bias_dev, s, sms) : launch_gemm2w<false>(ma, mb, mc, M, N, K, bias_dev, s, sms);
    if (act) {
      EpiBiasF16<true>::Params p{bias_dev};
      return launch_gemm2<EpiBiasF16<true>>(ma, mb, mc, M, N, K, p, s, sms);
    }
    EpiBiasF16<false>::Params p{bias_dev};
    return launch_gemm2<EpiBiasF16<false>>(ma, mb, mc, M, N, K, p, s, sms);
  }
  if (block_n == 128) return test_gemm_bn<128>(a16_dev, w16_dev, bias_dev, out16_dev, M, N, K, act, s, sms);
  return fail(B200MDM_EINVAL, "block_n must be 512 (CTA pair), 513 (CTA pair, W-resident) or 128 (single CTA)");
}

// Host-only: the dispatch decision of launch_gemm2_bias and the tile ownership of the W-resident order (the same
// arithmetic gemm2w_f16_tcgen05 does on the device), for the CPU tests.
extern "C" int b200mdm_test_gemm2_plan(int32_t M, int32_t N, int32_t K, int32_t num_sms, int32_t* plan_out, int32_t* tile_owner) {
  if (M <= 0 || N <= 0 || K <= 0 || num_sms < 2 || !plan_out) return fail(B200MDM_EINVAL, "bad argument");
  const int tiles_m = (M + GEMM2_TILE_M - 1) / GEMM2_TILE_M, tiles_n = (N + GEMM2_BLOCK_N - 1) / GEMM2_BLOCK_N;
  const int tiles = tiles_m * tiles_n, max_clusters = num_sms / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  const bool can = K <= GEMM2W_KB_MAX * GEMM_BLOCK_K && tiles_n <= clusters;
  plan_out[0] = gemm2w_pays(M, N, K, num_sms) ? 1 : 0;
  plan_out[1] = clusters;
  plan_out[2] = (tiles + clusters - 1) / clusters;
  plan_out[3] = -1;
  if (tile_owner)
    for (int i = 0; i < tiles; ++i) tile_owner[i] = -1;
  if (can) {
    int rounds = 0;
    for (int c = 0; c < clusters; ++c) {
      const int n_blk = c % tiles_n, m_first = c / tiles_n, m_step = (clusters - n_blk + tiles_n - 1) / tiles_n;
      int mine = 0;
      for (int m_blk = m_first; m_blk < tiles_m; m_blk += m_step, ++mine)
        if (tile_owner) {
          int32_t& o = tile_owner[m_blk * tiles_n + n_blk];
          o = (o == -1) ? c : -2;   // -2: two owners (never happens; the test checks)
        }
      rounds = mine > rounds ? mine : rounds;
    }
    plan_out[3] = rounds;
  }
  return B200MDM_OK;
}

extern "C" int b200mdm_test_attention(const void* qkv16_dev, void* out16_dev, const int32_t* kvlen_dev,
                                      int32_t n_samples, int32_t S, int32_t d, int32_t impl, void* stream) {
  if (!qkv16_dev || !out16_dev || !kvlen_dev || n_samples <= 0 || S <= 0) return fail(B200MDM_EINVAL, "bad argument");
  TRY(init_kernel_attrs());
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (impl != 0) return fail(B200MDM_EINVAL, "impl 0 (tcgen05) is the only attention kernel");
  if (S > ATC_MAX_KEYS) return fail(B200MDM_EINVAL, "tcgen05 attention handles at most %d tokens", ATC_MAX_KEYS);
  AttnMaps am;
  TRY(make_attn_maps(&am, static_cast<const __half*>(qkv16_dev), static_cast<__half*>(out16_dev), n_samples, S, d));
  return launch_attention_tc(am, kvlen_dev, n_samples, S, d, d / ATC_DH, s);
}

extern "C" int b200mdm_test_cross_attention(const void* q16_dev, const void* kv16_dev, const unsigned char* mask_dev,
                                            void* out16_dev, int32_t n_samples, int32_t S, int32_t n_tokens, int32_t ld_kv,
                                            void* stream) {
  const int d = 512;
  if (!q16_dev || !kv16_dev || !mask_dev || !out16_dev || n_samples <= 0 || S <= 0 || n_tokens <= 0 || n_tokens > 64 ||
      ld_kv < 2 * d || ld_kv % 8)
    return fail(B200MDM_EINVAL, "bad argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float sl2 = 1.4426950408889634f / sqrtf(128.0f);
  const dim3 cg(d / 128, n_samples), cb(128);
  const __half* q = static_cast<const __half*>(q16_dev);
  const __half* kv = static_cast<const __half*>(kv16_dev);
  __half* o = static_cast<__half*>(out16_dev);
  if (n_tokens <= 16) CUDA_TRY(launch_k(cross_attention_kernel<2>, cg, cb, 0, s, q, kv, mask_dev, o, S, n_tokens, d, ld_kv, sl2));
  else if (n_tokens <= 32) CUDA_TRY(launch_k(cross_attention_kernel<4>, cg, cb, 0, s, q, kv, mask_dev, o, S, n_tokens, d, ld_kv, sl2));
  else CUDA_TRY(launch_k(cross_attention_kernel<8>, cg, cb, 0, s, q, kv, mask_dev, o, S, n_tokens, d, ld_kv, sl2));
  return B200MDM_OK;
}

extern "C" int b200mdm_test_qkv_attention(const void* h16_dev, int32_t ld, const void* wqkv16_dev, const float* bqkv_dev,
                                          void* out16_dev, const int32_t* kvlen_dev, int32_t n_samples, int32_t S,
                                          void* stream) {
  if (!h16_dev || !wqkv16_dev || !bqkv_dev || !out16_dev || !kvlen_dev || n_samples <= 0 || S <= 0 || S > 256 || ld < 512 || ld % 8)
    return fail(B200MDM_EINVAL, "bad argument");
  TRY(init_kernel_attrs());
  int dev = 0, sms = 148;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CUtensorMap mh, mw128, mw64, mo;
  TRY(make_map_3d(&mh, h16_dev, n_samples, S, 512, ld, 128));
  TRY(make_map(&mw128, wqkv16_dev, 1536, 512, 512, 128));
  TRY(make_map(&mw64, wqkv16_dev, 1536, 512, 512, 64));
  TRY(make_map_3d(&mo, out16_dev, n_samples, S, 512, 512, 32));
  return launch_qkv_attention(mh, mw128, mw64, mo, bqkv_dev, kvlen_dev, n_samples, S, static_cast<cudaStream_t>(stream), sms);
}

extern "C" int b200mdm_test_gemm_resid_ln(const void* a16_dev, const void* w16_dev, const float* bias_dev,
                                          const float* gamma_dev, const float* beta_dev, void* hres16_dev, int32_t M,
                                          int32_t K, void* stream) {
  if (!a16_dev || !w16_dev || !bias_dev || !gamma_dev || !beta_dev || !hres16_dev || M <= 0 || K <= 0 || K % 8)
    return fail(B200MDM_EINVAL, "bad argument");
  TRY(init_kernel_attrs());
  int dev = 0, sms = 148;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CUtensorMap ma, mb, mr;
  TRY(make_map(&ma, a16_dev, M, K, K, GEMM_BLOCK_M));
  TRY(make_map(&mb, w16_dev, GLN_D, K, K, 256));
  TRY(make_map_res(&mr, hres16_dev, M, GLN_D));
  return launch_gemm_resid_ln(ma, mb, mr, M, K, bias_dev, gamma_dev, beta_dev, static_cast<cudaStream_t>(stream), sms);
}

// Debug aid (not part of the public header): device buffer of 32 int64 that receives clock64 stamps of the fused
// residual+LayerNorm kernel (block 0, first epilogue warp): tile start, accumulator ready, pass 1 done, stats done, pass 2 done.
extern "C" int b200mdm_debug_trace(long long* dev_buf) {
  CUDA_TRY(cudaMemcpyToSymbol(g_gemm2_trace, &dev_buf, sizeof(dev_buf)));
  return B200MDM_OK;
}

// ------------------------------------------------------------------------------------------------ post-processing
extern "C" int b200mdm_recover_from_ric(const float* data_dev, int64_t stride_b, int64_t stride_f, int64_t stride_t,
                                        const float* mean_dev, const float* std_dev, float* out_dev, int64_t ostride_b,
                                        int64_t ostride_t, int64_t ostride_c, int32_t batch, int32_t nframes,
                                        int32_t njoints, void* stream) {
  if (!data_dev || !out_dev || batch <= 0 || nframes <= 0 || njoints < 2) return fail(B200MDM_EINVAL, "bad argument");
  if ((mean_dev == nullptr) != (std_dev == nullptr)) return fail(B200MDM_EINVAL, "mean and std come together");
  const size_t smem = static_cast<size_t>(nframes) * 7 * sizeof(float);
  if (smem > 48 * 1024) return fail(B200MDM_ENOTIMPL, "recover_from_ric: %d frames exceed the single-CTA scan", nframes);
  RicArgs a;
  a.x = data_dev; a.xb = stride_b; a.xf = stride_f; a.xt = stride_t;
  a.mean = mean_dev; a.std = std_dev;
  a.out = out_dev; a.ob = ostride_b; a.ot = ostride_t; a.oc = ostride_c;
  a.T = nframes; a.joints = njoints;
  recover_from_ric_kernel<<<batch, 256, smem, static_cast<cudaStream_t>(stream)>>>(a);
  CUDA_TRY(cudaGetLastError());
  return B200MDM_OK;
}
