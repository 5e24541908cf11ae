// Memory-bound kernels of the FACT hot path and the fp32 CUDA-core GEMM used for the tiny embedding
// projections and as the debug cross-check of the tcgen05 path.
//   layernorm_split : Norm (mint/core/base_models.py:22-31) fused with the fp32 -> bf16 hi/lo operand split
//   pack_weight     : Keras [in,out] fp32 kernel -> K-major bf16 hi/lo [out,in]
//   gemm_f32        : LinearEmbedding + PositionEmbedding (base_models.py:130-156) and debug GEMMs
//   head_rows       : output Dense on one row per sample (base_models.py:200, fact_model.py:128)
//   mse             : FACTModel.loss (fact_model.py:143-148)
#include "fact_internal.h"
#include "fact_ptx.cuh"

namespace fact {

// ------------------------------------------------------------------------------------------- error plumbing
static thread_local char g_err[512] = "";
thread_local long long g_launch_count = 0;
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return FACT_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------- LayerNorm + split
// One warp per row, row kept in registers (d <= 1024, d % 4 == 0); two-pass mean / biased variance, eps 1e-5.
template <bool NORM>
__global__ void __launch_bounds__(256) ln_split_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, bf16* __restrict__ hi,
                                                       bf16* __restrict__ lo, int rows, int d) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  pdl_trigger();
  pdl_wait();
  if (row >= rows) return;
  float4 v[8];
  ln_row_load<false>(x + static_cast<size_t>(row) * d, d >> 2, lane, v);
  ln_row_finish<NORM>(v, gamma, beta, hi + static_cast<size_t>(row) * d, lo ? lo + static_cast<size_t>(row) * d : nullptr,
                      d, lane);
}

// ------------------------------------------------------------------------------------------- weight packing
// w [k_in, n_out] fp32 row-major  ->  hi/lo [n_out, k_in] bf16 (transpose through a padded shared tile)
__global__ void __launch_bounds__(256) pack_weight_kernel(const float* __restrict__ w, bf16* __restrict__ hi,
                                                          bf16* __restrict__ lo, int k_in, int n_out, int ld) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, n = n0 + tx;
    tile[r][tx] = (k < k_in && n < n_out) ? w[static_cast<size_t>(k) * n_out + n] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int n = n0 + r, k = k0 + tx;
    if (n < n_out && k < k_in) {
      bf16 h, l;
      split_bf16(tile[tx][r], h, l);
      hi[static_cast<size_t>(n) * ld + k] = h;
      if (lo) lo[static_cast<size_t>(n) * ld + k] = l;
    }
  }
}

// every dense kernel of the model in one launch (the training step repacks all of them after the optimizer update)
constexpr int PACK_MAX = 80;
struct PackTable {
  const float* w[PACK_MAX];
  bf16* hi[PACK_MAX];
  bf16* lo[PACK_MAX];
  int k_in[PACK_MAX], n_out[PACK_MAX];
  int tile0[PACK_MAX + 1];  // first 32 x 32 tile of tensor i in the flat grid
  int count;
};
__global__ void __launch_bounds__(256) pack_weights_kernel(const __grid_constant__ PackTable t) {
  __shared__ float tile[32][33];
  int idx = 0;
  while (idx + 1 < t.count && static_cast<int>(blockIdx.x) >= t.tile0[idx + 1]) ++idx;
  const int k_in = t.k_in[idx], n_out = t.n_out[idx];
  const int local = blockIdx.x - t.tile0[idx], tiles_n = (n_out + 31) / 32;
  const int k0 = (local / tiles_n) * 32, n0 = (local % tiles_n) * 32;
  const float* __restrict__ w = t.w[idx];
  bf16* __restrict__ hi = t.hi[idx];
  bf16* __restrict__ lo = t.lo[idx];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, n = n0 + tx;
    tile[r][tx] = (k < k_in && n < n_out) ? w[static_cast<size_t>(k) * n_out + n] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int n = n0 + r, k = k0 + tx;
    if (n < n_out && k < k_in) {
      bf16 h, l;
      split_bf16(tile[tx][r], h, l);
      hi[static_cast<size_t>(n) * k_in + k] = h;
      if (lo) lo[static_cast<size_t>(n) * k_in + k] = l;
    }
  }
}

// ------------------------------------------------------------------------------------------- fp32 SIMT GEMM
struct SimtArgs {
  // A operand: either fp32 (a_f32) or split bf16 (a_hi [+ a_lo]); row r lives at
  //   base + (r / a_seq) * a_batch_stride + (start + r % a_seq) * lda      (a_seq == 0: base + r * lda)
  const float* a_f32;
  const bf16* a_hi;
  const bf16* a_lo;
  long long a_batch_stride;
  int a_seq;
  const int* step_ptr;
  int lda;
  const float* w;  // Keras layout [k, n]
  int m, n, k;
  // epilogue
  int kind;
  float* out_f32;
  bf16* out_hi;
  bf16* out_lo;
  int ldo;
  const float* bias;
  const float* resid;
  int ldr;
  float scale;
  int scale_cols;
  int seq_in, seq_out, seq_off;
  const float* pos;  // [pos_seq, n] added to row (r % pos_seq), or NULL
  int pos_seq;
};

// TM x TN tile (64x64 or 128x128), 16-deep K slices, 256 threads x (TM/16 x TN/16) outputs each; the big tile is
// used for the embedding projections at batch >= 8 (8x8 register blocking: 64 FMA per 16 shared loads).
template <int TM, int TN>
__global__ void __launch_bounds__(256) gemm_f32_kernel(SimtArgs p) {
  constexpr int RM = TM / 16, RN = TN / 16;
  __shared__ float As[16][TM + 4];
  __shared__ float Ws[16][TN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int start = p.step_ptr ? *p.step_ptr : 0;
  float acc[RM][RN];
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < p.k; k0 += 16) {
    for (int e = threadIdx.x; e < TM * 16; e += 256) {
      const int r = e >> 4, kk = e & 15;  // A: k fastest -> coalesced along the row
      const int row = m0 + r, k = k0 + kk;
      float a = 0.f;
      if (row < p.m && k < p.k) {
        const size_t off = p.a_seq ? static_cast<size_t>(row / p.a_seq) * p.a_batch_stride +
                                         static_cast<size_t>(start + row % p.a_seq) * p.lda + k
                                   : static_cast<size_t>(row) * p.lda + k;
        if (p.a_f32) a = p.a_f32[off];
        else a = __bfloat162float(p.a_hi[off]) + (p.a_lo ? __bfloat162float(p.a_lo[off]) : 0.f);
      }
      As[kk][r] = a;
    }
    for (int e = threadIdx.x; e < 16 * TN; e += 256) {
      const int kk = e / TN, c = e % TN;
      const int k = k0 + kk, col = n0 + c;
      Ws[kk][c] = (k < p.k && col < p.n) ? p.w[static_cast<size_t>(k) * p.n + col] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[RM], w[RN];
      // strided ownership (row ty + 16 i, column tx + 16 j): conflict-free shared reads, coalesced global stores
#pragma unroll
      for (int i = 0; i < RM; ++i) a[i] = As[kk][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < RN; ++j) w[j] = Ws[kk][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < RM; ++i)
#pragma unroll
        for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    const int row = m0 + ty + 16 * i;
    if (row >= p.m) continue;
    const int orow = p.seq_in ? (row / p.seq_in) * p.seq_out + p.seq_off + row % p.seq_in : row;
#pragma unroll
    for (int j = 0; j < RN; ++j) {
      const int col = n0 + tx + 16 * j;
      if (col >= p.n) continue;
      float x = acc[i][j];
      if (p.kind == FACT_EPI_SPLIT) {
        if (col < p.scale_cols) x *= p.scale;
      } else if (p.bias) {
        x += p.bias[col];
      }
      if (p.pos) x += p.pos[static_cast<size_t>(row % p.pos_seq) * p.n + col];
      if (p.kind == FACT_EPI_BIAS_GELU_SPLIT) x = gelu_tanh(x);
      if (p.kind == FACT_EPI_BIAS_GELU_SAVE) {
        const size_t oz = static_cast<size_t>(orow) * p.ldo + col;
        p.out_lo[oz] = __float2bfloat16_rn(x);
        p.out_hi[oz] = __float2bfloat16_rn(gelu_tanh(x));
        continue;
      }
      if (p.kind == FACT_EPI_BIAS_RESID_F32) x += p.resid[static_cast<size_t>(row) * p.ldr + col];
      const size_t o = static_cast<size_t>(orow) * p.ldo + col;
      if (p.kind == FACT_EPI_SPLIT || p.kind == FACT_EPI_BIAS_GELU_SPLIT) {
        bf16 h, l;
        split_bf16(x, h, l);
        p.out_hi[o] = h;
        if (p.out_lo) p.out_lo[o] = l;
      } else {
        p.out_f32[o] = x;
      }
    }
  }
}

// LinearEmbedding at decode batch sizes (a few hundred rows, K = 225 / 35): the tiled kernel above puts the whole
// problem on ~26 blocks that each walk K in 15 synchronised steps (51 us at batch 1, on the critical path of every
// AR frame).  Here a block owns 8 rows x 64 columns and its 256 threads split K four ways, so ~200 blocks run
// ~60-long FMA chains with coalesced weight loads; the four partial sums meet in shared memory in a fixed order.
constexpr int ER_ROWS = 8, ER_COLS = 64, ER_KG = 4;
__global__ void __launch_bounds__(256) embed_rows_kernel(SimtArgs p) {
  extern __shared__ float er_smem[];   // [ER_ROWS][k] inputs, then [ER_KG - 1][ER_ROWS][ER_COLS] partials
  float* xs = er_smem;
  float* part = er_smem + ER_ROWS * p.k;
  const int tx = threadIdx.x & (ER_COLS - 1), kg = threadIdx.x / ER_COLS;
  const int m0 = blockIdx.y * ER_ROWS, col = blockIdx.x * ER_COLS + tx;
  pdl_trigger();
  pdl_wait();   // the step counter and the motion history row of the previous frame come from the previous graph launch
  const int start = p.step_ptr ? *p.step_ptr : 0;
  for (int e = threadIdx.x; e < ER_ROWS * p.k; e += 256) {
    const int r = e / p.k, k = e % p.k, row = m0 + r;
    float a = 0.f;
    if (row < p.m)
      a = p.a_f32[static_cast<size_t>(row / p.a_seq) * p.a_batch_stride +
                  static_cast<size_t>(start + row % p.a_seq) * p.lda + k];
    xs[e] = a;
  }
  __syncthreads();
  const int kper = (p.k + ER_KG - 1) / ER_KG;
  const int k0 = kg * kper, k1 = min(p.k, k0 + kper);
  float acc[ER_ROWS];
#pragma unroll
  for (int r = 0; r < ER_ROWS; ++r) acc[r] = 0.f;
  if (col < p.n) {
#pragma unroll 8
    for (int k = k0; k < k1; ++k) {
      const float w = __ldg(p.w + static_cast<size_t>(k) * p.n + col);
#pragma unroll
      for (int r = 0; r < ER_ROWS; ++r) acc[r] = fmaf(xs[r * p.k + k], w, acc[r]);
    }
  }
  if (kg > 0) {
#pragma unroll
    for (int r = 0; r < ER_ROWS; ++r) part[((kg - 1) * ER_ROWS + r) * ER_COLS + tx] = acc[r];
  }
  __syncthreads();
  if (kg == 0 && col < p.n) {
    const float b = p.bias ? p.bias[col] : 0.f;
#pragma unroll
    for (int r = 0; r < ER_ROWS; ++r) {
      const int row = m0 + r;
      if (row >= p.m) break;
      float x = acc[r];
#pragma unroll
      for (int g = 0; g < ER_KG - 1; ++g) x += part[(g * ER_ROWS + r) * ER_COLS + tx];
      x += b;
      if (p.pos) x += p.pos[static_cast<size_t>(row % p.pos_seq) * p.n + col];
      p.out_f32[static_cast<size_t>(row) * p.ldo + col] = x;
    }
  }
}

static int launch_simt(const SimtArgs& p, cudaStream_t st) {
  if (p.a_f32 && p.a_seq > 0 && p.kind == FACT_EPI_BIAS_F32 && p.seq_in == 0 && p.m <= 1024 && p.k <= 1024) {
    dim3 grid((p.n + ER_COLS - 1) / ER_COLS, (p.m + ER_ROWS - 1) / ER_ROWS);
    const size_t smem = (static_cast<size_t>(ER_ROWS) * p.k + (ER_KG - 1) * ER_ROWS * ER_COLS) * sizeof(float);
    FACT_CUDA_CHECK(launch_k(embed_rows_kernel, grid, dim3(256), smem, st, true, p));
    FACT_LAUNCH_CHECK("embed_rows_kernel launch");
    return FACT_OK;
  }
  if (p.m >= 1024 && p.n >= 128) {
    dim3 grid((p.n + 127) / 128, (p.m + 127) / 128);
    gemm_f32_kernel<128, 128><<<grid, 256, 0, st>>>(p);
  } else {
    dim3 grid((p.n + 63) / 64, (p.m + 63) / 64);
    gemm_f32_kernel<64, 64><<<grid, 256, 0, st>>>(p);
  }
  FACT_LAUNCH_CHECK("gemm_f32_kernel launch");
  return FACT_OK;
}

static void fill_epi(SimtArgs& p, const fact_gemm_epilogue* e) {
  p.kind = e->kind;
  p.out_f32 = e->out_f32;
  p.out_hi = static_cast<bf16*>(e->out_hi);
  p.out_lo = static_cast<bf16*>(e->out_lo);
  p.ldo = e->ldo;
  p.bias = e->bias;
  p.resid = e->resid;
  p.ldr = e->ldr;
  p.scale = e->scale;
  p.scale_cols = e->scale_cols;
  p.seq_in = e->seq_in;
  p.seq_out = e->seq_out;
  p.seq_off = e->seq_off;
  p.pos = nullptr;
  p.pos_seq = 1;
}

static int check_epi(const fact_gemm_epilogue* e) {
  FACT_REQUIRE(e != nullptr, FACT_ERR_BAD_SHAPE, "null epilogue");
  const bool split_out = e->kind == FACT_EPI_SPLIT || e->kind == FACT_EPI_BIAS_GELU_SPLIT ||
                         e->kind == FACT_EPI_BIAS_GELU_SAVE;
  FACT_REQUIRE(e->kind >= 0 && e->kind <= 4, FACT_ERR_UNSUPPORTED, "epilogue kind %d not available on the CUDA-core GEMM", e->kind);
  FACT_REQUIRE(split_out ? e->out_hi != nullptr : e->out_f32 != nullptr, FACT_ERR_BAD_SHAPE,
               "epilogue output buffer missing");
  FACT_REQUIRE(e->kind != FACT_EPI_BIAS_RESID_F32 || e->resid, FACT_ERR_BAD_SHAPE, "resid epilogue needs resid");
  FACT_REQUIRE(e->resid_rows == 0, FACT_ERR_UNSUPPORTED, "resid_rows is a tensor-path (fact_gemm) option");
  return FACT_OK;
}

// gemm on split-bf16 activations with the fp32 Keras-layout weight (FACT_MODE_FP32_SIMT); internal
int gemm_simt_split(const void* a_hi, const void* a_lo, int lda, const float* w_keras, int m, int n, int k,
                    const fact_gemm_epilogue* epi, cudaStream_t st) {
  int rc = check_epi(epi);
  if (rc) return rc;
  FACT_REQUIRE(a_hi && w_keras, FACT_ERR_BAD_SHAPE, "gemm_simt_split: null operand (fp32 weights not provided?)");
  SimtArgs p{};
  p.a_hi = static_cast<const bf16*>(a_hi);
  p.a_lo = static_cast<const bf16*>(a_lo);
  p.lda = lda;
  p.w = w_keras;
  p.m = m;
  p.n = n;
  p.k = k;
  fill_epi(p, epi);
  return launch_simt(p, st);
}

// ------------------------------------------------------------------------------------------- head on one row / sample
constexpr int HR_COLS = 32, HR_KG = 8;
__global__ void __launch_bounds__(256) head_rows_kernel(const float* __restrict__ x, long long row_stride,
                                                        const float* __restrict__ w, const float* __restrict__ bias,
                                                        float* __restrict__ out, long long out_batch_stride,
                                                        const int* __restrict__ step_ptr, int d, int out_dim) {
  // block (b, c) = clip b, 32 output columns; 8 groups of 32 threads split the reduction dimension (100-long FMA
  // chains with coalesced weight loads) and meet in shared memory in a fixed order.  One block per clip with 4
  // groups was 21 us at batch 1 (800 / 4 dependent loads per thread on a single SM).
  extern __shared__ float xs[];          // [d] input row, then [HR_KG - 1][HR_COLS] partials
  const int b = blockIdx.x;
  const int grp = threadIdx.x / HR_COLS, t = threadIdx.x % HR_COLS;
  const float* xr = x + static_cast<size_t>(b) * row_stride * d;
  pdl_trigger();
  pdl_wait();
  for (int i = threadIdx.x; i < d; i += blockDim.x) xs[i] = xr[i];
  __syncthreads();
  float* part = xs + d;
  const int step = step_ptr ? *step_ptr : 0;
  const int kper = (d + HR_KG - 1) / HR_KG;
  const int k0 = grp * kper, k1 = min(d, k0 + kper);
  const int j = blockIdx.y * HR_COLS + t;
  float acc = 0.f;
  if (j < out_dim) {
#pragma unroll 10
    for (int k = k0; k < k1; ++k) acc = fmaf(xs[k], __ldg(w + static_cast<size_t>(k) * out_dim + j), acc);
  }
  if (grp > 0) part[(grp - 1) * HR_COLS + t] = acc;
  __syncthreads();
  if (grp == 0 && j < out_dim) {
#pragma unroll
    for (int g = 0; g < HR_KG - 1; ++g) acc += part[g * HR_COLS + t];
    out[static_cast<size_t>(b) * out_batch_stride + static_cast<size_t>(step) * out_dim + j] = acc + bias[j];
  }
}

// ------------------------------------------------------------------------------------------- MSE
__global__ void __launch_bounds__(256) mse_partial_kernel(const float* __restrict__ target,
                                                          const float* __restrict__ pred, float* __restrict__ partial,
                                                          int batch, int t_len, int n, int od) {
  const long long total = static_cast<long long>(batch) * t_len * od;
  float s = 0.f;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += 256ll * gridDim.x) {
    const int j = static_cast<int>(i % od);
    const long long bt = i / od;
    const int t = static_cast<int>(bt % t_len), b = static_cast<int>(bt / t_len);
    const float df = target[i] - pred[(static_cast<size_t>(b) * n + t) * od + j];
    s = fmaf(df, df, s);
  }
  __shared__ float red[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; ++i) tsum += red[i];
    partial[blockIdx.x] = tsum;
  }
}
__global__ void __launch_bounds__(256) mse_final_kernel(const float* __restrict__ partial, int nparts, float* loss,
                                                        float inv_total) {
  __shared__ float red[8];
  float s = 0.f;
  for (int i = threadIdx.x; i < nparts; i += 256) s += partial[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; ++i) tsum += red[i];
    *loss = tsum * inv_total;
  }
}
__global__ void __launch_bounds__(256) mse_grad_kernel(const float* __restrict__ target,
                                                       const float* __restrict__ pred, float* __restrict__ dpred,
                                                       int batch, int t_len, int n, int od, float coef) {
  const long long total = static_cast<long long>(batch) * n * od;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += 256ll * gridDim.x) {
    const int j = static_cast<int>(i % od);
    const long long bt = i / od;
    const int t = static_cast<int>(bt % n), b = static_cast<int>(bt / n);
    dpred[i] = t < t_len ? coef * (pred[i] - target[(static_cast<size_t>(b) * t_len + t) * od + j]) : 0.f;
  }
}

__global__ void step_set_kernel(int* p, int v) { *p = v; }
__global__ void step_inc_kernel(int* p) {
  pdl_trigger();
  pdl_wait();
  *p += 1;
}

int step_set(int* p, int v, cudaStream_t st) {
  step_set_kernel<<<1, 1, 0, st>>>(p, v);
  FACT_LAUNCH_CHECK("step_set_kernel");
  return FACT_OK;
}
int step_inc(int* p, cudaStream_t st) {
  FACT_CUDA_CHECK(launch_k(step_inc_kernel, dim3(1), dim3(1), 0, st, true, p));
  FACT_LAUNCH_CHECK("step_inc_kernel");
  return FACT_OK;
}

}  // namespace fact

using namespace fact;

extern "C" int fact_abi_version(void) { return FACT_ABI_VERSION; }
extern "C" long long fact_launch_count(void) { return g_launch_count; }
extern "C" const char* fact_last_error(void) { return g_err; }

extern "C" int fact_layernorm_split(const float* x, const float* gamma, const float* beta, void* y_hi, void* y_lo,
                                    int rows, int d, void* stream) {
  FACT_REQUIRE(x && y_hi, FACT_ERR_BAD_SHAPE, "fact_layernorm_split: null buffer");
  FACT_REQUIRE(rows > 0 && d > 0 && d % 4 == 0 && d <= 1024, FACT_ERR_BAD_SHAPE,
               "fact_layernorm_split: need 0 < d <= 1024, d %% 4 == 0 (rows=%d d=%d)", rows, d);
  FACT_REQUIRE((gamma == nullptr) == (beta == nullptr), FACT_ERR_BAD_SHAPE, "gamma and beta go together");
  FACT_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y_hi) & 7) == 0,
               FACT_ERR_BAD_ALIGN, "fact_layernorm_split: x must be 16-B, y 8-B aligned");
  const int grid = (rows + 7) / 8;
  cudaStream_t st = as_stream(stream);
  const float* no_f = nullptr;
  if (gamma)
    FACT_CUDA_CHECK(launch_k(ln_split_kernel<true>, dim3(grid), dim3(256), 0, st, true, x, gamma, beta,
                             static_cast<bf16*>(y_hi), static_cast<bf16*>(y_lo), rows, d));
  else
    FACT_CUDA_CHECK(launch_k(ln_split_kernel<false>, dim3(grid), dim3(256), 0, st, true, x, no_f, no_f,
                             static_cast<bf16*>(y_hi), static_cast<bf16*>(y_lo), rows, d));
  FACT_LAUNCH_CHECK("ln_split_kernel launch");
  return FACT_OK;
}

namespace fact {
// ---- tensor-core embedding (large batches): LinearEmbedding as a tcgen05 GEMM on split inputs
// x rows -> bf16 hi / lo with row pitch kp (>= f, multiple of 8; the pad is never read: the TMA map is f wide).
// Row r = clip r / n_tok, frame start + r % n_tok (the AR window: start = *step_ptr), as in the CUDA-core path.
__global__ void __launch_bounds__(256) embed_prep_kernel(const float* __restrict__ x, long long batch_stride,
                                                         const int* __restrict__ step_ptr, bf16* __restrict__ hi,
                                                         bf16* __restrict__ lo, int rows, int n_tok, int f, int kp) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int start = step_ptr ? *step_ptr : 0;
  const float* src = x + static_cast<size_t>(row / n_tok) * batch_stride + static_cast<size_t>(start + row % n_tok) * f;
  for (int c = lane; c < f; c += 32) {
    bf16 h, l;
    split_bf16(src[c], h, l);
    hi[static_cast<size_t>(row) * kp + c] = h;
    if (lo) lo[static_cast<size_t>(row) * kp + c] = l;
  }
}

int embed_prep(const float* x, long long batch_stride, const int* step_ptr, void* hi, void* lo, int rows, int n_tok,
               int f, int kp, cudaStream_t st) {
  embed_prep_kernel<<<(rows + 7) / 8, 256, 0, st>>>(x, batch_stride, step_ptr, static_cast<bf16*>(hi),
                                                    static_cast<bf16*>(lo), rows, n_tok, f, kp);
  FACT_LAUNCH_CHECK("embed_prep_kernel launch");
  return FACT_OK;
}

// w [k_in, n_out] fp32 -> hi / lo [n_out, ld] bf16 (ld >= k_in)
int pack_weight_ld(const float* w, void* hi, void* lo, int k_in, int n_out, int ld, cudaStream_t st) {
  dim3 grid((n_out + 31) / 32, (k_in + 31) / 32);
  pack_weight_kernel<<<grid, 256, 0, st>>>(w, static_cast<bf16*>(hi), static_cast<bf16*>(lo), k_in, n_out, ld);
  FACT_LAUNCH_CHECK("pack_weight_kernel launch");
  return FACT_OK;
}

}  // namespace fact
using namespace fact;

extern "C" int fact_pack_weight(const float* w_keras, void* hi, void* lo, int k_in, int n_out, void* stream) {
  FACT_REQUIRE(w_keras && hi && k_in > 0 && n_out > 0, FACT_ERR_BAD_SHAPE, "fact_pack_weight: bad arguments");
  dim3 grid((n_out + 31) / 32, (k_in + 31) / 32);
  pack_weight_kernel<<<grid, 256, 0, as_stream(stream)>>>(w_keras, static_cast<bf16*>(hi), static_cast<bf16*>(lo),
                                                          k_in, n_out, k_in);
  FACT_LAUNCH_CHECK("pack_weight_kernel launch");
  return FACT_OK;
}

extern "C" int fact_pack_weights(const float* const* w_keras, void* const* hi, void* const* lo, const int* k_in,
                                 const int* n_out, int count, void* stream) {
  FACT_REQUIRE(w_keras && hi && k_in && n_out && count > 0, FACT_ERR_BAD_SHAPE, "fact_pack_weights: bad arguments");
  for (int base = 0; base < count; base += PACK_MAX) {
    PackTable t{};
    t.count = count - base < PACK_MAX ? count - base : PACK_MAX;
    int tiles = 0;
    for (int i = 0; i < t.count; ++i) {
      const int j = base + i;
      FACT_REQUIRE(w_keras[j] && hi[j] && k_in[j] > 0 && n_out[j] > 0, FACT_ERR_BAD_SHAPE,
                   "fact_pack_weights: bad entry %d", j);
      t.w[i] = w_keras[j];
      t.hi[i] = static_cast<bf16*>(hi[j]);
      t.lo[i] = lo ? static_cast<bf16*>(lo[j]) : nullptr;
      t.k_in[i] = k_in[j];
      t.n_out[i] = n_out[j];
      t.tile0[i] = tiles;
      tiles += ((k_in[j] + 31) / 32) * ((n_out[j] + 31) / 32);
    }
    t.tile0[t.count] = tiles;
    pack_weights_kernel<<<tiles, 256, 0, as_stream(stream)>>>(t);
    FACT_LAUNCH_CHECK("pack_weights_kernel launch");
  }
  return FACT_OK;
}

extern "C" int fact_gemm_f32(const float* a, int lda, const float* w_keras, int m, int n, int k,
                             const fact_gemm_epilogue* epi, void* stream) {
  int rc = check_epi(epi);
  if (rc) return rc;
  FACT_REQUIRE(a && w_keras && m > 0 && n > 0 && k > 0, FACT_ERR_BAD_SHAPE, "fact_gemm_f32: bad arguments");
  SimtArgs p{};
  p.a_f32 = a;
  p.lda = lda;
  p.w = w_keras;
  p.m = m;
  p.n = n;
  p.k = k;
  fill_epi(p, epi);
  return launch_simt(p, as_stream(stream));
}

extern "C" int fact_embed(const float* x, long long x_batch_stride, const int* step_ptr, const float* w,
                          const float* bias, const float* pos, float* y, int batch, int n_tok, int f, int d,
                          void* stream) {
  FACT_REQUIRE(x && w && bias && pos && y, FACT_ERR_BAD_SHAPE, "fact_embed: null buffer");
  FACT_REQUIRE(batch > 0 && n_tok > 0 && f > 0 && d > 0, FACT_ERR_BAD_SHAPE, "fact_embed: bad shape");
  SimtArgs p{};
  p.a_f32 = x;
  p.a_batch_stride = x_batch_stride;
  p.a_seq = n_tok;
  p.step_ptr = step_ptr;
  p.lda = f;
  p.w = w;
  p.m = batch * n_tok;
  p.n = d;
  p.k = f;
  p.kind = FACT_EPI_BIAS_F32;
  p.out_f32 = y;
  p.ldo = d;
  p.bias = bias;
  p.pos = pos;
  p.pos_seq = n_tok;
  return launch_simt(p, as_stream(stream));
}

extern "C" int fact_head_rows(const float* x, long long row_stride, const float* w_keras, const float* bias,
                              float* out, long long out_batch_stride, const int* step_ptr, int batch, int d,
                              int out_dim, void* stream) {
  FACT_REQUIRE(x && w_keras && bias && out, FACT_ERR_BAD_SHAPE, "fact_head_rows: null buffer");
  FACT_REQUIRE(batch > 0 && d > 0 && d <= 8192 && out_dim > 0, FACT_ERR_BAD_SHAPE, "fact_head_rows: bad shape");
  const dim3 grid(batch, (out_dim + HR_COLS - 1) / HR_COLS);
  FACT_CUDA_CHECK(launch_k(head_rows_kernel, grid, dim3(256), (d + (HR_KG - 1) * HR_COLS) * sizeof(float),
                           as_stream(stream), true, x, row_stride, w_keras, bias, out, out_batch_stride, step_ptr, d,
                           out_dim));
  FACT_LAUNCH_CHECK("head_rows_kernel launch");
  return FACT_OK;
}

extern "C" int fact_mse(const float* target, const float* pred, float* loss, float* dpred, float* partial, int batch,
                        int t_len, int n, int out_dim, float loss_scale, void* stream) {
  FACT_REQUIRE(target && pred && loss && partial, FACT_ERR_BAD_SHAPE, "fact_mse: null buffer");
  FACT_REQUIRE(batch > 0 && t_len > 0 && t_len <= n && out_dim > 0, FACT_ERR_BAD_SHAPE, "fact_mse: bad shape");
  const long long total = static_cast<long long>(batch) * t_len * out_dim;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > 1024) grid = 1024;
  cudaStream_t st = as_stream(stream);
  mse_partial_kernel<<<grid, 256, 0, st>>>(target, pred, partial, batch, t_len, n, out_dim);
  FACT_LAUNCH_CHECK("mse_partial_kernel launch");
  mse_final_kernel<<<1, 256, 0, st>>>(partial, grid, loss, 1.0f / static_cast<float>(total));
  FACT_LAUNCH_CHECK("mse_final_kernel launch");
  if (dpred) {
    const long long all = static_cast<long long>(batch) * n * out_dim;
    int g2 = static_cast<int>((all + 255) / 256);
    if (g2 > 4096) g2 = 4096;
    mse_grad_kernel<<<g2, 256, 0, st>>>(target, pred, dpred, batch, t_len, n, out_dim,
                                        2.0f * loss_scale / static_cast<float>(total));
    FACT_LAUNCH_CHECK("mse_grad_kernel launch");
  }
  return FACT_OK;
}

// Training windows out of a device-resident dataset (fact_gather_windows).  blockIdx.z picks the output (0 motion
// input, 1 target, 2 audio input), blockIdx.y the clip; each window is one contiguous span of len * dim floats in both
// the arena and the output, so the blocks along x copy it with coalesced loads and stores.
__global__ void __launch_bounds__(256) gather_windows_kernel(
    const float* __restrict__ motion, int motion_dim, const float* __restrict__ audio, int audio_dim,
    const long long* __restrict__ motion_row, const long long* __restrict__ audio_row, int motion_len,
    int target_shift, int target_len, int audio_len, float* __restrict__ motion_out, float* __restrict__ target_out,
    float* __restrict__ audio_out) {
  const int b = blockIdx.y;
  const float* src;
  float* dst;
  long long n;
  if (blockIdx.z == 0) {
    n = static_cast<long long>(motion_len) * motion_dim;
    src = motion + motion_row[b] * motion_dim;
    dst = motion_out + b * n;
  } else if (blockIdx.z == 1) {
    n = static_cast<long long>(target_len) * motion_dim;
    src = motion + (motion_row[b] + target_shift) * motion_dim;
    dst = target_out + b * n;
  } else {
    n = static_cast<long long>(audio_len) * audio_dim;
    src = audio + audio_row[b] * audio_dim;
    dst = audio_out + b * n;
  }
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i];
}

extern "C" int fact_gather_windows(const float* motion, int motion_dim, const float* audio, int audio_dim,
                                   const long long* motion_row, const long long* audio_row, int batch, int motion_len,
                                   int target_shift, int target_len, int audio_len, float* motion_out,
                                   float* target_out, float* audio_out, void* stream) {
  FACT_REQUIRE(motion && audio && motion_row && audio_row && motion_out && target_out && audio_out, FACT_ERR_BAD_SHAPE,
               "fact_gather_windows: null buffer");
  FACT_REQUIRE(batch > 0 && batch <= 65535 && motion_dim > 0 && audio_dim > 0, FACT_ERR_BAD_SHAPE,
               "fact_gather_windows: bad shape (batch %d, motion_dim %d, audio_dim %d)", batch, motion_dim, audio_dim);
  FACT_REQUIRE(motion_len > 0 && target_len > 0 && audio_len > 0 && target_shift >= 0, FACT_ERR_BAD_SHAPE,
               "fact_gather_windows: bad window (motion_len %d, target_shift %d, target_len %d, audio_len %d)",
               motion_len, target_shift, target_len, audio_len);
  long long span = static_cast<long long>(motion_len) * motion_dim;
  if (static_cast<long long>(audio_len) * audio_dim > span) span = static_cast<long long>(audio_len) * audio_dim;
  if (static_cast<long long>(target_len) * motion_dim > span) span = static_cast<long long>(target_len) * motion_dim;
  long long blocks = (span + 1023) / 1024;                       // ~4 floats per thread on the longest window
  if (blocks > 1024) blocks = 1024;
  gather_windows_kernel<<<dim3(static_cast<unsigned>(blocks), batch, 3), 256, 0, as_stream(stream)>>>(
      motion, motion_dim, audio, audio_dim, motion_row, audio_row, motion_len, target_shift, target_len, audio_len,
      motion_out, target_out, audio_out);
  FACT_LAUNCH_CHECK("gather_windows_kernel launch");
  return FACT_OK;
}
