// Exact fp32 (SIMT) scoring kernels: the fp32 flavour of get_sim_scores (method/model.py:307-329)
// and of the clip-scale head, used (a) as the exact drop-in path, (b) to rescore the bf16 GEMM's
// top-K candidates, (c) for the key-clip dot products of the attention table.
//
// One tiled "dots" kernel: block = 64 query rows x kRows corpus rows of ONE video, K = D streamed
// in 32-wide chunks through shared memory (padded stride 36 words: conflict-free LDS.128),
// 256 threads, each thread 2 query rows x kRows/8 corpus rows.  Two epilogues (max/argmax, store).
// The clip-scale flavour lives in dkd_exact_tc.cu (tensor cores).
#include <cuda_fp16.h>

#include "dkd_common.cuh"

namespace dkd {

constexpr int kTM = 64;      // query rows per block
constexpr int kKC = 32;      // K chunk
constexpr int kLd = kKC + 4; // padded smem stride (words); 36 % 32 == 4 -> 8 rows hit 32 banks

enum { EPI_MAX = 0, EPI_STORE = 2 };

struct DotsParams {
  const float* q;          // query rows
  int64_t q_video_stride;  // elements added per video (0: queries shared by all videos)
  int M;                   // number of query rows (dense) / upper bound (CSR)
  const float* x;          // (Nv, R, D)
  int R, D, T;
  const uint8_t* mask;     // (Nv, R) or null
  float* out_max;
  int32_t* out_arg;
  int64_t ld_out;
  float* out_rows;         // EPI_MAX optional (M, R, Nv); EPI_STORE: E (Nv, M, T)
  int Nv;
  const int32_t* vid_ptr;  // CSR (optional)
  const int32_t* q_list;
};

template <int kRows, int kEpi>
__global__ void __launch_bounds__(256)
dots_kernel(const DotsParams p) {
  constexpr int kJ = kRows / 8;
  __shared__ __align__(16) float sQ[kTM * kLd];
  __shared__ __align__(16) float sX[kRows * kLd];

  const int n = blockIdx.x;
  const int tile = blockIdx.y;
  int e0 = 0, count = p.M;
  if (p.vid_ptr) {
    e0 = p.vid_ptr[n];
    count = p.vid_ptr[n + 1] - e0;
  }
  const int r0 = tile * kTM;
  if (r0 >= count) return;
  const int tid = threadIdx.x;
  const int tm = tid >> 3;  // 0..31 -> query rows tm, tm + 32
  const int ti = tid & 7;   // corpus rows ti + 8 j
  const float* qbase = p.q + (int64_t)n * p.q_video_stride;
  const float* xbase = p.x + (int64_t)n * p.R * p.D;

  float acc[2][kJ];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int j = 0; j < kJ; ++j) acc[a][j] = 0.f;

  // global row of each of the 2 float4 slots this thread loads for the Q tile
  // Q tile: 64 rows x 8 float4 = 512 float4 -> 2 per thread
  int64_t qrow[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int r = (tid + t * 256) >> 3;
    const int lr = r0 + r;
    if (lr < count) qrow[t] = p.q_list ? (int64_t)p.q_list[e0 + lr] : (int64_t)lr;
    else qrow[t] = -1;
  }

  for (int kc = 0; kc < p.D; kc += kKC) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int idx = tid + t * 256;
      const int r = idx >> 3, c4 = idx & 7;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (qrow[t] >= 0) v = *reinterpret_cast<const float4*>(&qbase[qrow[t] * p.D + kc + c4 * 4]);
      *reinterpret_cast<float4*>(&sQ[r * kLd + c4 * 4]) = v;
    }
#pragma unroll
    for (int t = 0; t < kRows / 32; ++t) {
      const int idx = tid + t * 256;
      const int r = idx >> 3, c4 = idx & 7;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < p.R) v = *reinterpret_cast<const float4*>(&xbase[(int64_t)r * p.D + kc + c4 * 4]);
      *reinterpret_cast<float4*>(&sX[r * kLd + c4 * 4]) = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kKC; k += 4) {
      const float4 a0 = *reinterpret_cast<const float4*>(&sQ[tm * kLd + k]);
      const float4 a1 = *reinterpret_cast<const float4*>(&sQ[(tm + 32) * kLd + k]);
#pragma unroll
      for (int j = 0; j < kJ; ++j) {
        const float4 b = *reinterpret_cast<const float4*>(&sX[(ti + 8 * j) * kLd + k]);
        acc[0][j] = fmaf(a0.x, b.x, acc[0][j]);
        acc[0][j] = fmaf(a0.y, b.y, acc[0][j]);
        acc[0][j] = fmaf(a0.z, b.z, acc[0][j]);
        acc[0][j] = fmaf(a0.w, b.w, acc[0][j]);
        acc[1][j] = fmaf(a1.x, b.x, acc[1][j]);
        acc[1][j] = fmaf(a1.y, b.y, acc[1][j]);
        acc[1][j] = fmaf(a1.z, b.z, acc[1][j]);
        acc[1][j] = fmaf(a1.w, b.w, acc[1][j]);
      }
    }
    __syncthreads();
  }

  if constexpr (kEpi == EPI_STORE) {
    // E[n][m][row] = key[n][m] . clips[n][row]
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int lr = r0 + tm + 32 * a;
      if (lr >= count) continue;
#pragma unroll
      for (int j = 0; j < kJ; ++j) {
        const int row = ti + 8 * j;
        if (row < p.T) p.out_rows[((int64_t)n * p.M + lr) * p.T + row] = acc[a][j];
      }
    }
  } else {  // EPI_MAX
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int lr = r0 + tm + 32 * a;
      const bool live = lr < count;
      float bv = -INFINITY;
      int bi = 0x7fffffff;
#pragma unroll
      for (int j = 0; j < kJ; ++j) {
        const int row = ti + 8 * j;
        if (row < p.R) {
          float v = acc[a][j];
          if (p.mask && p.mask[(int64_t)n * p.R + row] == 0) v = DKD_MASKED_SCORE;
          if (live && p.out_rows) {
            const int64_t m = p.q_list ? p.q_list[e0 + lr] : lr;
            p.out_rows[(m * p.R + row) * (int64_t)p.Nv + n] = v;
          }
          if (better(v, row, bv, bi)) { bv = v; bi = row; }
        }
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      if (live && ti == 0) {
        const int64_t o = p.vid_ptr ? (int64_t)(e0 + lr) : (int64_t)lr * p.ld_out + n;
        p.out_max[o] = bv;
        if (p.out_arg) p.out_arg[o] = bi;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Frame-scale score + branch fusion.  8 lanes per (query, video) pair; block = 256 threads
// covers 32 queries x 8 videos; grid x = query tiles (fastest) so concurrent blocks share the
// same 8 videos' table slices in L2.
template <typename TT>
struct RowLoader;
template <>
struct RowLoader<float> {
  static __device__ __forceinline__ float dot(const float* a, const float* b, int D, int sub) {
    float acc = 0.f;
    for (int d = sub * 4; d < D; d += 32) {
      const float4 x = *reinterpret_cast<const float4*>(a + d);
      const float4 y = *reinterpret_cast<const float4*>(b + d);
      acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
      acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
    return acc;
  }
};
__device__ __forceinline__ float fuse_branch(float clip, float frame, float wc, float wf, float wb) {
  // torch: w_clip * clip + w_frame * frame ; numpy: w_branch * branch   (no FMA contraction)
  const float br = __fadd_rn(__fmul_rn(wc, clip), __fmul_rn(wf, frame));
  return __fmul_rn(wb, br);
}

template <typename TT>
__global__ void __launch_bounds__(256)
frame_fuse_kernel(const TT* __restrict__ q, const TT* __restrict__ table,
                  const float* __restrict__ clip, const int32_t* __restrict__ key_clip, int M, int Nv,
                  int P, int D, int64_t ld, float wc, float wf, float wb, int accumulate,
                  float* __restrict__ out_frame, float* __restrict__ fused) {
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  const int n = blockIdx.y * 8 + (grp & 7);
  const int mrow = grp >> 3;  // 0..3
  for (int it = 0; it < 8; ++it) {
    const int m = blockIdx.x * 32 + it * 4 + mrow;
    const bool live = (m < M) && (n < Nv);
    float acc = 0.f;
    int64_t o = 0;
    if (live) {
      o = (int64_t)m * ld + n;
      int k = key_clip[o];
      k = k < 0 ? 0 : (k >= P ? P - 1 : k);
      acc = RowLoader<TT>::dot(q + (int64_t)m * D, table + ((int64_t)n * P + k) * D, D, sub);
    }
#pragma unroll
    for (int s = 4; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (live && sub == 0) {
      if (out_frame) out_frame[o] = acc;
      if (fused) {
        const float v = fuse_branch(clip[o], acc, wc, wf, wb);
        fused[o] = accumulate ? __fadd_rn(fused[o], v) : v;
      }
    }
  }
}

// fp16 flavour of the dense gather (the approximate pass of the bf16 path).  An 8-lane group owns ONE query
// for a chunk of videos: its 8 x (D/8) query halves stay in registers, per video only the key clip's table
// row is fetched (768 B at D = 384: six 128-byte wavefronts per pair).  Products are formed and summed four
// at a time in half2 (HFMA2), each 4-product partial sum is widened and accumulated in fp32.  Eight videos
// are processed per step and their 8 x 8 lane partials reduced by a 7-shuffle transpose, so that lane j ends
// with the frame score of video n0 + j: the (clip, key clip) loads and the fused stores are 32-byte runs.
// Register budget of the gather (round-2 A/B inside the whole step, profiles/r2_ab_gather.md): with plain
// __launch_bounds__(256) ptxas settles at 70 registers and keeps ~9 row loads in flight per lane: 2.75 ms per step (two
// launches); telling it that 3 blocks per SM are enough (<= 85 registers) lets it keep more loads in flight at the same
// occupancy: 2.03 ms.  4 blocks (<= 64 registers) 2.44, 1 block (212 registers, every load hoisted) 3.30; loading the
// rows of 2 / 4 videos explicitly before consuming them (DKD_FF_BATCH) 2.13 / 2.03 at 3 blocks.
#ifndef DKD_FF_BATCH
#define DKD_FF_BATCH 1      // videos whose table rows are loaded before any of them is consumed
#endif
#ifndef DKD_FF_MINBLOCKS
#define DKD_FF_MINBLOCKS 3
#endif
#define DKD_FF_BOUNDS __launch_bounds__(256, DKD_FF_MINBLOCKS)
template <int kC>  // D = 64 * kC
__global__ void DKD_FF_BOUNDS
frame_fuse_h_kernel(const __half* __restrict__ q, const __half* __restrict__ table,
                    const float* __restrict__ clip, const int32_t* __restrict__ key_clip, int M, int Nv,
                    int P, int64_t ld, float wc, float wf, float wb, int accumulate, int vchunk,
                    float* __restrict__ out_frame, float* __restrict__ fused) {
  constexpr int D = 64 * kC;
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  const int m = blockIdx.x * 32 + grp;
  const bool live_m = m < M;
  const int mm = live_m ? m : M - 1;
  const int n_begin = blockIdx.y * vchunk;
  const int n_end = min(Nv, n_begin + vchunk);
  uint4 qv[kC];
#pragma unroll
  for (int i = 0; i < kC; ++i) qv[i] = *reinterpret_cast<const uint4*>(q + (int64_t)mm * D + 64 * i + 8 * sub);
  const unsigned gmask = 0xffffffffu;                   // all groups of a warp run the same trip counts
  for (int n0 = n_begin; n0 < n_end; n0 += 8) {
    const int nj = n0 + sub;
    const bool valid = nj < n_end;
    const int64_t oj = (int64_t)mm * ld + (valid ? nj : n_begin);
    int kk = key_clip[oj];
    kk = kk < 0 ? 0 : (kk >= P ? P - 1 : kk);
    float part[8];
#pragma unroll
    for (int j0 = 0; j0 < 8; j0 += DKD_FF_BATCH) {
      uint4 t[DKD_FF_BATCH][kC];
#pragma unroll
      for (int b = 0; b < DKD_FF_BATCH; ++b) {
        const int k = __shfl_sync(gmask, kk, j0 + b, 8);
        const int n = min(n0 + j0 + b, n_end - 1);
        const __half* row = table + ((int64_t)n * P + k) * D + 8 * sub;
#pragma unroll
        for (int i = 0; i < kC; ++i) t[b][i] = __ldg(reinterpret_cast<const uint4*>(row + 64 * i));
      }
#pragma unroll
      for (int b = 0; b < DKD_FF_BATCH; ++b) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < kC; ++i) {
          const __half2* tp = reinterpret_cast<const __half2*>(&t[b][i]);
          const __half2* qp = reinterpret_cast<const __half2*>(&qv[i]);
          __half2 s2 = __hmul2(tp[0], qp[0]);
          s2 = __hfma2(tp[1], qp[1], s2);
          s2 = __hfma2(tp[2], qp[2], s2);
          s2 = __hfma2(tp[3], qp[3], s2);
          const float2 f = __half22float2(s2);
          acc += f.x + f.y;
        }
        part[j0 + b] = acc;
      }
    }
    // transpose-reduce: after the three rounds lane `sub` holds the total of pair `sub`
    float r4[4], r2[2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = (sub & 4) ? part[j] : part[j + 4];
      const float keep = (sub & 4) ? part[j + 4] : part[j];
      r4[j] = keep + __shfl_xor_sync(gmask, send, 4);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = (sub & 2) ? r4[j] : r4[j + 2];
      const float keep = (sub & 2) ? r4[j + 2] : r4[j];
      r2[j] = keep + __shfl_xor_sync(gmask, send, 2);
    }
    const float send = (sub & 1) ? r2[0] : r2[1];
    const float keep = (sub & 1) ? r2[1] : r2[0];
    const float frame = keep + __shfl_xor_sync(gmask, send, 1);
    if (live_m && valid) {
      if (out_frame) out_frame[oj] = frame;
      if (fused) {
        const float v = fuse_branch(clip[oj], frame, wc, wf, wb);
        fused[oj] = accumulate ? __fadd_rn(fused[oj], v) : v;
      }
    }
  }
}

// Bulk-copy flavour of the fp16 gather.  Same mapping (an 8-lane group owns one query, its query halves in registers;
// eight videos per step reduced by the 7-shuffle transpose), but the key clips' table rows travel by cp.async.bulk
// (768 B per row at D = 384, one instruction of one lane, completion on an mbarrier) into a per-group ring of 8 row
// slots in shared memory instead of through 48 LDG.128 per row into registers: the bytes in flight per SM are set by
// the 196 KB of ring (8 rows x 32 groups) instead of by the registers left over next to the query (~110 KB at 70
// registers x 768 threads).  The gather is latency bound — L2 at ~52 % of its peak in the register version
// (profiles/r2_ncu_step.md) — so more bytes in flight looked like the lever.
// MEASURED (round 2, same box, whole step): 6.13 ms per step against 2.51 ms for the register version — one 768-byte
// bulk copy per (query, video) pair (23.7 M per launch) is bound by the copy engine's per-request cost, not by bytes in
// flight.  Kept as the record of that experiment; compiled only with -DDKD_FF_BULK=1.
#ifndef DKD_FF_BULK
#define DKD_FF_BULK 0
#endif
#if DKD_FF_BULK
__device__ __forceinline__ uint32_t ff_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int kC>
__global__ void __launch_bounds__(256, 1)
frame_fuse_h_bulk_kernel(const __half* __restrict__ q, const __half* __restrict__ table,
                         const float* __restrict__ clip, const int32_t* __restrict__ key_clip, int M, int Nv,
                         int P, int64_t ld, float wc, float wf, float wb, int accumulate, int vchunk,
                         float* __restrict__ out_frame, float* __restrict__ fused) {
  constexpr int D = 64 * kC;
  constexpr uint32_t kRowBytes = D * 2;
  extern __shared__ __align__(128) uint8_t ff_smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(ff_smem + 32 * 8 * kRowBytes);     // [group][slot]
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  const int m = blockIdx.x * 32 + grp;
  const bool live_m = m < M;
  const int mm = live_m ? m : M - 1;
  const int n_begin = blockIdx.y * vchunk;
  const int n_end = min(Nv, n_begin + vchunk);
  uint8_t* ring = ff_smem + (size_t)grp * 8 * kRowBytes;
  uint64_t* gbar = bars + grp * 8;
  if (sub == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ff_smem_u32(&gbar[j])));
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  uint4 qv[kC];
#pragma unroll
  for (int i = 0; i < kC; ++i) qv[i] = *reinterpret_cast<const uint4*>(q + (int64_t)mm * D + 64 * i + 8 * sub);
  const unsigned gmask = 0xffu << ((threadIdx.x & 31) & ~7);          // the 8 lanes of this group
  auto issue = [&](int j, int n, int k) {                              // lane 0 of the group: row of video n -> slot j
    const __half* src = table + ((int64_t)n * P + k) * D;
    const uint32_t bar = ff_smem_u32(&gbar[j]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kRowBytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(ff_smem_u32(ring + (size_t)j * kRowBytes)), "l"(src), "r"(kRowBytes), "r"(bar) : "memory");
  };
  auto load_key = [&](int n0) {
    const int nj = min(n0 + sub, n_end - 1);
    int kk = key_clip[(int64_t)mm * ld + nj];
    return kk < 0 ? 0 : (kk >= P ? P - 1 : kk);
  };
  int kk = load_key(n_begin);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = __shfl_sync(gmask, kk, j, 8);
    if (sub == 0) issue(j, min(n_begin + j, n_end - 1), k);
  }
  uint32_t phase = 0;
  for (int n0 = n_begin; n0 < n_end; n0 += 8) {
    const bool more = n0 + 8 < n_end;
    const int kk_next = more ? load_key(n0 + 8) : 0;
    float part[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t bar = ff_smem_u32(&gbar[j]);
      uint32_t ok = 0, spins = 0;
      while (!ok) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(phase) : "memory");
        if (!ok && ++spins > (1u << 26)) __trap();                    // a protocol bug traps instead of hanging the GPU
      }
      const uint8_t* row = ring + (size_t)j * kRowBytes + 16 * sub;
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < kC; ++i) {
        const uint4 t = *reinterpret_cast<const uint4*>(row + 128 * i);
        const __half2* tp = reinterpret_cast<const __half2*>(&t);
        const __half2* qp = reinterpret_cast<const __half2*>(&qv[i]);
        __half2 s2 = __hmul2(tp[0], qp[0]);
        s2 = __hfma2(tp[1], qp[1], s2);
        s2 = __hfma2(tp[2], qp[2], s2);
        s2 = __hfma2(tp[3], qp[3], s2);
        const float2 f = __half22float2(s2);
        acc += f.x + f.y;
      }
      part[j] = acc;
      __syncwarp(gmask);                                               // every lane has read slot j
      if (more) {
        const int k = __shfl_sync(gmask, kk_next, j, 8);
        if (sub == 0) issue(j, min(n0 + 8 + j, n_end - 1), k);
      }
    }
    phase ^= 1u;
    // transpose-reduce: after the three rounds lane `sub` holds the total of pair `sub`
    float r4[4], r2[2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = (sub & 4) ? part[j] : part[j + 4];
      const float keep = (sub & 4) ? part[j + 4] : part[j];
      r4[j] = keep + __shfl_xor_sync(gmask, send, 4);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = (sub & 2) ? r4[j] : r4[j + 2];
      const float keep = (sub & 2) ? r4[j + 2] : r4[j];
      r2[j] = keep + __shfl_xor_sync(gmask, send, 2);
    }
    const float send = (sub & 1) ? r2[0] : r2[1];
    const float keep = (sub & 1) ? r2[1] : r2[0];
    const float frame = keep + __shfl_xor_sync(gmask, send, 1);
    const int nj = n0 + sub;
    if (live_m && nj < n_end) {
      const int64_t oj = (int64_t)mm * ld + nj;
      if (out_frame) out_frame[oj] = frame;
      if (fused) {
        const float v = fuse_branch(clip[oj], frame, wc, wf, wb);
        fused[oj] = accumulate ? __fadd_rn(fused[oj], v) : v;
      }
    }
  }
}

#endif  // DKD_FF_BULK

// CSR flavour (exact rescoring of candidates): one 8-lane group per CSR entry.
// kD > 0: the row length is a compile-time constant and the body is fully unrolled (query row + table row: 2 x kD / 32
// float4 per lane) — the kernel is a latency-bound random gather of 1.5 KB rows from HBM / L2, so the loads in flight
// per SM set its speed; the summation order is that of the generic loop (bit-identical results).
// Round-2 A/B (whole step, two launches, ms): generic loop at 40 registers 0.75; the fully unrolled D = 384 body at
// 3 / 4 / 5 blocks per SM 0.79 / 0.67 / 0.65; forcing all 24 loads ahead of the arithmetic (116 registers, 2 blocks) 0.96.
#ifndef DKD_CSR_MINBLOCKS
#define DKD_CSR_MINBLOCKS 5    // 0: plain __launch_bounds__(256) and the generic loop (round-1 kernel)
#endif
#if DKD_CSR_MINBLOCKS > 0
#define DKD_CSR_BOUNDS __launch_bounds__(256, DKD_CSR_MINBLOCKS)
#else
#define DKD_CSR_BOUNDS __launch_bounds__(256)
#endif
// kDetail: also write this branch's (key clip, clip score bits, frame score bits) to payload[slot[e] * C + c0 ..]
// (dkd_frame_fuse_csr_detail); the kDetail = false instantiations are the kernels of dkd_frame_fuse_csr.
template <int kD, bool kDetail = false>
__global__ void DKD_CSR_BOUNDS
frame_fuse_csr_kernel(const float* __restrict__ q, const float* __restrict__ table,
                      const float* __restrict__ clip, const int32_t* __restrict__ key_clip,
                      const int32_t* __restrict__ vid_ptr, const int32_t* __restrict__ q_list,
                      const int32_t* __restrict__ slot, int Nv, int P, int D, float wc, float wf,
                      float wb, int accumulate, float* __restrict__ cand_scores, int64_t dense_ld,
                      uint32_t* __restrict__ payload = nullptr, int C = 0, int c0 = 0) {
  // dense_ld > 0: clip / key_clip are dense (M, Nv) matrices indexed by (query, video) instead of per-entry arrays
  const int n = blockIdx.x;
  const int e0 = vid_ptr[n], e1 = vid_ptr[n + 1];
  const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
  for (int base = e0 + blockIdx.y * 32; base < e1; base += gridDim.y * 32) {
    const int e = base + grp;
    const bool live = e < e1;
    float acc = 0.f;
    int64_t ce = e;
    int k = 0;
    if (live) {
      if (dense_ld > 0) ce = (int64_t)q_list[e] * dense_ld + n;
      k = key_clip[ce];
      k = k < 0 ? 0 : (k >= P ? P - 1 : k);
      const float* a = q + (int64_t)q_list[e] * D;
      const float* b = table + ((int64_t)n * P + k) * D;
      if (kD > 0) {
        constexpr int kN = kD > 0 ? kD / 32 : 1;
        float4 x[kN], y[kN];
#pragma unroll
        for (int i = 0; i < kN; ++i) {
          x[i] = __ldg(reinterpret_cast<const float4*>(a + sub * 4 + 32 * i));
          y[i] = __ldg(reinterpret_cast<const float4*>(b + sub * 4 + 32 * i));
        }
#ifdef DKD_CSR_BARRIER
        asm volatile("" ::: "memory");                    // keep every load of the entry ahead of the arithmetic
#endif
#pragma unroll
        for (int i = 0; i < kN; ++i) {
          acc = fmaf(x[i].x, y[i].x, acc); acc = fmaf(x[i].y, y[i].y, acc);
          acc = fmaf(x[i].z, y[i].z, acc); acc = fmaf(x[i].w, y[i].w, acc);
        }
      } else {
        acc = RowLoader<float>::dot(a, b, D, sub);
      }
    }
#pragma unroll
    for (int s = 4; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (live && sub == 0) {
      const float v = fuse_branch(clip[ce], acc, wc, wf, wb);
      const int sl = slot[e];
      cand_scores[sl] = accumulate ? __fadd_rn(cand_scores[sl], v) : v;
      if constexpr (kDetail) {
        uint32_t* pd = payload + (int64_t)sl * C + c0;
        pd[0] = (uint32_t)k;
        pd[1] = __float_as_uint(clip[ce]);
        pd[2] = __float_as_uint(acc);
      }
    }
  }
}

__global__ void fuse_scores_kernel(const float* __restrict__ a, const float* __restrict__ b, float wa,
                                   float wb, float* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __fadd_rn(__fmul_rn(wa, a[i]), __fmul_rn(wb, b[i]));
}

}  // namespace dkd

using namespace dkd;

template <int kRows, int kEpi>
static int launch_dots(const DotsParams& p, int Nv, int tiles, cudaStream_t st) {
  if (Nv == 0 || tiles == 0) return DKD_OK;
  dim3 grid(Nv, tiles);
  dots_kernel<kRows, kEpi><<<grid, 256, 0, st>>>(p);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_score_max_f32(const float* qn, int32_t M, const float* xn, int32_t Nv, int32_t R,
                                 int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg,
                                 int64_t ld_out, float* out_rows, const int32_t* vid_ptr,
                                 const int32_t* q_list, void* stream) {
  if (!qn || !xn || !out_max || M < 0 || Nv < 0) return DKD_ERR_ARG;
  if ((vid_ptr == nullptr) != (q_list == nullptr)) return DKD_ERR_ARG;
  if (R <= 0 || R > 128 || D <= 0 || D % kKC != 0) return DKD_ERR_SHAPE;
  if (!vid_ptr && ld_out < Nv) return DKD_ERR_ARG;
  if (M == 0 || Nv == 0) return DKD_OK;
  if (M > 65535 * kTM) return DKD_ERR_SHAPE;
  DotsParams p{};
  p.q = qn; p.q_video_stride = 0; p.M = M; p.x = xn; p.R = R; p.D = D; p.T = 0; p.mask = mask;
  p.out_max = out_max; p.out_arg = out_arg; p.ld_out = ld_out; p.out_rows = out_rows;
  p.Nv = Nv; p.vid_ptr = vid_ptr; p.q_list = q_list;
  const int tiles = (M + kTM - 1) / kTM;
  if (R <= 32) return launch_dots<32, EPI_MAX>(p, Nv, tiles, (cudaStream_t)stream);
  if (R <= 64) return launch_dots<64, EPI_MAX>(p, Nv, tiles, (cudaStream_t)stream);
  return launch_dots<128, EPI_MAX>(p, Nv, tiles, (cudaStream_t)stream);
}

extern "C" int dkd_key_clip_dots(const float* key, const float* clips, int32_t Nv, int32_t L, int32_t T,
                                 int32_t D, float* E, void* stream) {
  if (!key || !clips || !E || Nv < 0) return DKD_ERR_ARG;
  if (L <= 0 || T <= 0 || T > 32 || D <= 0 || D % kKC != 0) return DKD_ERR_SHAPE;
  if (Nv == 0) return DKD_OK;
  DotsParams p{};
  p.q = key; p.q_video_stride = (int64_t)L * D; p.M = L; p.x = clips; p.R = T; p.D = D; p.T = T;
  p.out_rows = E; p.Nv = Nv;
  return launch_dots<32, EPI_STORE>(p, Nv, (L + kTM - 1) / kTM, (cudaStream_t)stream);
}

extern "C" int dkd_frame_fuse(const void* q, const void* table, int32_t is_f16, const float* clip_scores,
                              const int32_t* key_clip, int32_t M, int32_t Nv, int32_t P, int32_t D,
                              int64_t ld, float w_clip, float w_frame, float w_branch, int32_t accumulate,
                              float* out_frame, float* fused, void* stream) {
  if (!q || !table || !key_clip || M < 0 || Nv < 0 || (!out_frame && !fused)) return DKD_ERR_ARG;
  if (fused && !clip_scores) return DKD_ERR_ARG;
  if (D <= 0 || D % 64 != 0 || P <= 0) return DKD_ERR_SHAPE;
  if (ld < Nv) return DKD_ERR_ARG;
  if (M == 0 || Nv == 0) return DKD_OK;
  dim3 grid((M + 31) / 32, (Nv + 7) / 8);
  if (grid.y > 65535) return DKD_ERR_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  if (is_f16) {
    if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(table)) & 15) return DKD_ERR_ALIGN;
    const int vchunk = 32;                                 // videos per block: amortises the query registers
    dim3 gh((M + 31) / 32, (Nv + vchunk - 1) / vchunk);
    const __half* qh = (const __half*)q;
    const __half* th = (const __half*)table;
#if DKD_FF_BULK
    if (D == 384) {   // bulk-copy ring (see frame_fuse_h_bulk_kernel); other widths keep the register version
      const int vch = 64;
      dim3 gb((M + 31) / 32, (Nv + vch - 1) / vch);
      const size_t smem = (size_t)32 * 8 * 768 + 32 * 8 * sizeof(uint64_t);
      DKD_CUDA_TRY(cudaFuncSetAttribute(frame_fuse_h_bulk_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      frame_fuse_h_bulk_kernel<6><<<gb, 256, smem, st>>>(qh, th, clip_scores, key_clip, M, Nv, P, ld, w_clip, w_frame,
                                                         w_branch, accumulate, vch, out_frame, fused);
      DKD_LAUNCH_CHECK();
      return DKD_OK;
    }
#endif
#define DKD_FF_H(C)                                                                                              \
  frame_fuse_h_kernel<C><<<gh, 256, 0, st>>>(qh, th, clip_scores, key_clip, M, Nv, P, ld, w_clip, w_frame,       \
                                             w_branch, accumulate, vchunk, out_frame, fused)
    switch (D / 64) {
      case 1: DKD_FF_H(1); break;
      case 2: DKD_FF_H(2); break;
      case 3: DKD_FF_H(3); break;
      case 4: DKD_FF_H(4); break;
      case 5: DKD_FF_H(5); break;
      case 6: DKD_FF_H(6); break;
      case 7: DKD_FF_H(7); break;
      case 8: DKD_FF_H(8); break;
      default: return DKD_ERR_SHAPE;
    }
#undef DKD_FF_H
  } else {
    frame_fuse_kernel<float><<<grid, 256, 0, st>>>((const float*)q, (const float*)table, clip_scores,
                                                   key_clip, M, Nv, P, D, ld, w_clip, w_frame, w_branch,
                                                   accumulate, out_frame, fused);
  }
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

template <bool kDetail>
static int launch_frame_fuse_csr(const float* q, const float* table, const float* clip_scores, const int32_t* key_clip,
                                 const int32_t* vid_ptr, const int32_t* q_list, const int32_t* slot, int32_t Nv,
                                 int32_t P, int32_t D, float w_clip, float w_frame, float w_branch, int32_t accumulate,
                                 float* cand_scores, int64_t dense_ld, uint32_t* payload, int32_t C, int32_t c0,
                                 void* stream) {
  if (!q || !table || !clip_scores || !key_clip || !vid_ptr || !q_list || !slot || !cand_scores || Nv < 0)
    return DKD_ERR_ARG;
  if (dense_ld != 0 && dense_ld < Nv) return DKD_ERR_ARG;
  if (D <= 0 || D % 32 != 0 || P <= 0) return DKD_ERR_SHAPE;
  if (Nv == 0) return DKD_OK;
  dim3 grid(Nv, 4);
  if (D == 384 && DKD_CSR_MINBLOCKS > 0)
    frame_fuse_csr_kernel<384, kDetail><<<grid, 256, 0, (cudaStream_t)stream>>>(
        q, table, clip_scores, key_clip, vid_ptr, q_list, slot, Nv, P, D, w_clip, w_frame, w_branch, accumulate,
        cand_scores, dense_ld, payload, C, c0);
  else
    frame_fuse_csr_kernel<0, kDetail><<<grid, 256, 0, (cudaStream_t)stream>>>(
        q, table, clip_scores, key_clip, vid_ptr, q_list, slot, Nv, P, D, w_clip, w_frame, w_branch, accumulate,
        cand_scores, dense_ld, payload, C, c0);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_frame_fuse_csr(const float* q, const float* table, const float* clip_scores,
                                  const int32_t* key_clip, const int32_t* vid_ptr, const int32_t* q_list,
                                  const int32_t* slot, int32_t Nv, int32_t P, int32_t D, float w_clip,
                                  float w_frame, float w_branch, int32_t accumulate, float* cand_scores,
                                  int64_t dense_ld, void* stream) {
  return launch_frame_fuse_csr<false>(q, table, clip_scores, key_clip, vid_ptr, q_list, slot, Nv, P, D, w_clip, w_frame,
                                      w_branch, accumulate, cand_scores, dense_ld, nullptr, 0, 0, stream);
}

extern "C" int dkd_frame_fuse_csr_detail(const float* q, const float* table, const float* clip_scores,
                                         const int32_t* key_clip, const int32_t* vid_ptr, const int32_t* q_list,
                                         const int32_t* slot, int32_t Nv, int32_t P, int32_t D, float w_clip,
                                         float w_frame, float w_branch, int32_t accumulate, float* cand_scores,
                                         int64_t dense_ld, uint32_t* payload, int32_t C, int32_t c0, void* stream) {
  if (!payload) return DKD_ERR_ARG;
  if (c0 < 0 || c0 + 3 > C) return DKD_ERR_SHAPE;
  return launch_frame_fuse_csr<true>(q, table, clip_scores, key_clip, vid_ptr, q_list, slot, Nv, P, D, w_clip, w_frame,
                                     w_branch, accumulate, cand_scores, dense_ld, payload, C, c0, stream);
}

extern "C" int dkd_fuse_scores(const float* a, const float* b, float wa, float wb, float* out, int64_t n,
                               void* stream) {
  if (!a || !b || !out || n < 0) return DKD_ERR_ARG;
  if (n == 0) return DKD_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  fuse_scores_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, b, wa, wb, out, n);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}
