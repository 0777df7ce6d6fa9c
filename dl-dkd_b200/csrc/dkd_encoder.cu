// Corpus-side encoder kernels (SURVEY section 8 f1: DLDKD.encode_context -> encode_input, method/model.py:215-243;
// LinearLayer / TrainablePositionalEncoding / BertAttention, method/model_components.py:269-312, :339-436).
//
// The linear layers run on the tcgen05 kind::tf32 x 3 pipeline (dkd_linear_exact, dkd_exact_umma.cu mode 4); this
// file holds what surrounds them:
//   dkd_row_stats        LayerNorm statistics of the raw frame features -> per-row (scale, shift) consumed by the
//                        projection GEMM's A-operand stager (the normalised features never exist in HBM)
//   dkd_layernorm_rows   LayerNorm over D <= 512 of (x [+ positional row] [+ residual]) — the two post-LN points of
//                        the block (after the projection + position table, after the attention output + residual)
//   dkd_mha_small        4-head self-attention over L <= 128 frames with the reference's additive -10000 key mask
//                        (model_components.py:420-422): scores, softmax and the weighted sum in one kernel per (video,
//                        head), fp32 throughout
#include "dkd_common.cuh"

namespace dkd {

// one warp per row: mean and 1/sqrt(var + eps) (biased variance, torch.nn.LayerNorm) -> (scale, shift) = (rstd, -mean*rstd)
__global__ void __launch_bounds__(256)
row_stats_kernel(const float* __restrict__ x, int64_t rows, int D, float eps, float2* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const float4* p = reinterpret_cast<const float4*>(x + row * D);
  const int n4 = D >> 2;
  float s = 0.f;
  for (int i = lane; i < n4; i += 32) { const float4 v = __ldg(p + i); s += (v.x + v.y) + (v.z + v.w); }
  s = warp_sum(s);
  const float mean = s / (float)D;
  float q = 0.f;
  for (int i = lane; i < n4; i += 32) {
    const float4 v = __ldg(p + i);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / (float)D + eps);
  if (lane == 0) out[row] = make_float2(rstd, -mean * rstd);
}

// one warp per row, D <= 512 (D % 4 == 0): y = LN(x + pos[row % L] + residual) * gamma + beta
__global__ void __launch_bounds__(256)
layernorm_rows_kernel(const float* __restrict__ x, int64_t x_ld, int64_t rows, int D, const float* __restrict__ gamma,
                      const float* __restrict__ beta, float eps, const float* __restrict__ residual, int64_t res_ld,
                      const float* __restrict__ pos, int L, float* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const int n4 = D >> 2;
  float4 v[4];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = lane + 32 * k;
    v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n4) {
      v[k] = __ldg(reinterpret_cast<const float4*>(x + row * x_ld) + i);
      if (pos) {
        const float4 p = __ldg(reinterpret_cast<const float4*>(pos + (row % L) * D) + i);
        v[k].x += p.x; v[k].y += p.y; v[k].z += p.z; v[k].w += p.w;
      }
      if (residual) {
        const float4 r = __ldg(reinterpret_cast<const float4*>(residual + row * res_ld) + i);
        v[k].x += r.x; v[k].y += r.y; v[k].z += r.z; v[k].w += r.w;
      }
      s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  }
  s = warp_sum(s);
  const float mean = s / (float)D;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (lane + 32 * k < n4) {
      const float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / (float)D + eps);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = lane + 32 * k;
    if (i < n4) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i);
      float4 o;
      o.x = (v[k].x - mean) * rstd * g.x + b.x; o.y = (v[k].y - mean) * rstd * g.y + b.y;
      o.z = (v[k].z - mean) * rstd * g.z + b.z; o.w = (v[k].w - mean) * rstd * g.w + b.w;
      reinterpret_cast<float4*>(out + row * D)[i] = o;
    }
  }
}

// Self-attention of one (video, head): qkv (Nv * L, ld) fp32 with the head's Q / K / V at column offsets
// q_off / k_off / v_off + head * dh.  K^T and V of the head live in shared memory; one warp owns 4 query rows at a time:
// scores over the L keys (lane = key, 4 keys per lane), + (1 - mask) * -10000, softmax, weighted sum over V
// (lane = output feature, dh <= 128).  out (Nv * L, out_ld) at column head * dh.
constexpr int kAttLmax = 128;
template <int kDh>
__global__ void __launch_bounds__(256)
mha_small_kernel(const float* __restrict__ qkv, int64_t ld, int q_off, int k_off, int v_off, const uint8_t* __restrict__ mask,
                 int L, int heads, float scale, float* __restrict__ out, int64_t out_ld) {
  extern __shared__ __align__(16) float smem_att[];
  float* sK = smem_att;                         // [L][kDh + 1]
  float* sV = sK + kAttLmax * (kDh + 1);        // [L][kDh]
  float* sP = sV + kAttLmax * kDh;              // [8 warps][L] probabilities of the warp's current row
  float* sQ = sP + 8 * kAttLmax;                // [8 warps][kDh]
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* base = qkv + (int64_t)n * L * ld;
  for (int i = threadIdx.x; i < L * kDh; i += 256) {
    const int l = i / kDh, d = i % kDh;
    sK[l * (kDh + 1) + d] = base[(int64_t)l * ld + k_off + h * kDh + d];
    sV[l * kDh + d] = base[(int64_t)l * ld + v_off + h * kDh + d];
  }
  __syncthreads();
  const uint8_t* mrow = mask ? mask + (int64_t)n * L : nullptr;
  for (int r = warp; r < L; r += 8) {
    for (int d = lane; d < kDh; d += 32) sQ[warp * kDh + d] = base[(int64_t)r * ld + q_off + h * kDh + d];
    __syncwarp();
    float sc[4];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = lane + 32 * j;
      float a = -INFINITY;
      if (l < L) {
        a = 0.f;
        const float* kr = sK + l * (kDh + 1);
        const float* qr = sQ + warp * kDh;
#pragma unroll 8
        for (int d = 0; d < kDh; ++d) a = fmaf(qr[d], kr[d], a);
        a = a * scale;
        if (mrow && mrow[l] == 0) a += -10000.0f;
      }
      sc[j] = a;
      mx = fmaxf(mx, a);
    }
    mx = warp_max(mx);
    float den = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = lane + 32 * j;
      const float e = l < L ? __expf(sc[j] - mx) : 0.f;
      sc[j] = e;
      den += e;
    }
    den = warp_sum(den);
    const float inv = 1.0f / den;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = lane + 32 * j;
      if (l < L) sP[warp * kAttLmax + l] = sc[j] * inv;
    }
    __syncwarp();
    for (int d = lane; d < kDh; d += 32) {
      float acc = 0.f;
      for (int l = 0; l < L; ++l) acc = fmaf(sP[warp * kAttLmax + l], sV[l * kDh + d], acc);
      out[((int64_t)n * L + r) * out_ld + h * kDh + d] = acc;
    }
    __syncwarp();
  }
}

}  // namespace dkd

using namespace dkd;

extern "C" int dkd_row_stats(const float* x, int64_t rows, int32_t D, float eps, float* scale_shift, void* stream) {
  if (!x || !scale_shift || rows < 0) return DKD_ERR_ARG;
  if (D <= 0 || D % 4 != 0) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(scale_shift)) & 15) return DKD_ERR_ALIGN;
  if (rows == 0) return DKD_OK;
  row_stats_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, rows, D, eps,
                                                                                 reinterpret_cast<float2*>(scale_shift));
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_layernorm_rows(const float* x, int64_t x_ld, int64_t rows, int32_t D, const float* gamma, const float* beta,
                                  float eps, const float* residual, int64_t res_ld, const float* pos, int32_t L, float* out,
                                  void* stream) {
  if (!x || !gamma || !beta || !out || rows < 0) return DKD_ERR_ARG;
  if (D <= 0 || D % 4 != 0 || D > 512 || (pos && L <= 0) || x_ld < D || x_ld % 4 != 0 || (residual && (res_ld < D || res_ld % 4 != 0)))
    return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(gamma) |
       reinterpret_cast<uintptr_t>(beta) | reinterpret_cast<uintptr_t>(residual) | reinterpret_cast<uintptr_t>(pos)) & 15)
    return DKD_ERR_ALIGN;
  if (rows == 0) return DKD_OK;
  layernorm_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, x_ld, rows, D, gamma, beta, eps,
                                                                                      residual, res_ld, pos, L > 0 ? L : 1, out);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

template <int kDh>
static int launch_mha(const float* qkv, int64_t ld, int q_off, int k_off, int v_off, const uint8_t* mask, int Nv, int L,
                      int heads, float scale, float* out, int64_t out_ld, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((size_t)kAttLmax * (kDh + 1) + (size_t)kAttLmax * kDh + 8 * kAttLmax + 8 * kDh);
  DKD_CUDA_TRY(cudaFuncSetAttribute(mha_small_kernel<kDh>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mha_small_kernel<kDh><<<(unsigned)(Nv * heads), 256, smem, st>>>(qkv, ld, q_off, k_off, v_off, mask, L, heads, scale, out,
                                                                  out_ld);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_mha_small(const float* qkv, int64_t ld, int32_t q_off, int32_t k_off, int32_t v_off, const uint8_t* mask,
                             int32_t Nv, int32_t L, int32_t heads, int32_t dh, float scale, float* out, int64_t out_ld,
                             void* stream) {
  if (!qkv || !out || Nv < 0 || heads <= 0) return DKD_ERR_ARG;
  if (L <= 0 || L > kAttLmax || (int64_t)Nv * heads > 0x7fffffffLL) return DKD_ERR_SHAPE;
  // every head's q / k / v columns inside a row of qkv, every head's output columns inside a row of out
  const int64_t width = (int64_t)heads * dh;
  const int64_t max_off = q_off > k_off ? (q_off > v_off ? q_off : v_off) : (k_off > v_off ? k_off : v_off);
  if (q_off < 0 || k_off < 0 || v_off < 0 || max_off + width > ld || out_ld < width) return DKD_ERR_SHAPE;
  if (Nv == 0) return DKD_OK;
  cudaStream_t st = (cudaStream_t)stream;
  switch (dh) {
    case 16: return launch_mha<16>(qkv, ld, q_off, k_off, v_off, mask, Nv, L, heads, scale, out, out_ld, st);
    case 32: return launch_mha<32>(qkv, ld, q_off, k_off, v_off, mask, Nv, L, heads, scale, out, out_ld, st);
    case 64: return launch_mha<64>(qkv, ld, q_off, k_off, v_off, mask, Nv, L, heads, scale, out, out_ld, st);
    case 96: return launch_mha<96>(qkv, ld, q_off, k_off, v_off, mask, Nv, L, heads, scale, out, out_ld, st);
    case 128: return launch_mha<128>(qkv, ld, q_off, k_off, v_off, mask, Nv, L, heads, scale, out, out_ld, st);
  }
  return DKD_ERR_SHAPE;
}
