// Moment localisation: the top-m non-overlapping clip windows of every listed (query, video) pair, ranked by the exact
// clip-scale curve (temporal non-maximum suppression over the P = T(T+1)/2 windows).
//
//   S_b(p(w, s)) = fl(run_b(s, w) * prop_scale_b[n, p])      run_b = d_b[s] + ... + d_b[s+w-1], sequential __fadd_rn
//   score(p)     = S_0(p)  (one branch)   |   fl(w0 * S_0(p)) + fl(w1 * S_1(p))  (two branches, dkd_fuse_scores order)
//   m rounds: pick the unsuppressed window of greatest score (lower p on equal scores), then suppress every window whose
//   temporal IoU with the pick, fl(inter / union) in clip units on [s, s + w), is above iou.
// d_b are the per-clip dots of dkd_clip_dots_list, so max_p S_b is the clip score of dkd_clip_score_f32 bit for bit.
// Replaces the clip-scale curve of get_clip_scale_scores (SURVEY §8 N3) that DLDKD.get_pred_from_raw_query reduces to
// its maximum: here the curve of every ranked hit is kept and reduced to m distinct moments.
//
// One block per video (or per chunk of its CSR run), the video's prop_scale row(s) in shared memory; one warp per entry:
//   curve   lane s runs the window sums of start s (w = 1 .. T - s) and writes the scores to the warp's 32 x 32 table
//           in shared memory; lane j then holds the windows p = j (mod 32): 17 values, slot k = p >> 5
//   rounds  lane-local best (slots in p order, strict >), a warp (value desc, p asc) argmax by shuffles, then an
//           integer suppression test per slot: fl(i / u) is non-increasing in u, so fl(i / u) > iou  <=>  u <= umax[i]
//           with umax tabulated once per block by __fdiv_rn — the same predicate, without a division per test
// Both loops are branch-free (selects, unconditional stores to padded rows): a branch per window measured 4.5 ms at
// TVR shape (1.09 M entries, two branches, m = 5) on a B200.
#include "dkd_common.cuh"

namespace dkd {

constexpr int kNmsWarps = 8;
constexpr int kNmsSlots = 17;                // ceil(528 / 32) windows per lane
constexpr int kNmsMaxP = 528;
constexpr int kNmsNone = 0x7fffffff;

template <bool kTwo>
__global__ void __launch_bounds__(kNmsWarps * 32)
moment_nms_kernel(const float* __restrict__ dots0, const float* __restrict__ scale0, const float* __restrict__ dots1,
                  const float* __restrict__ scale1, float w0, float w1, const int32_t* __restrict__ vid_ptr,
                  const int32_t* __restrict__ slot, int T, int m, float iou, int32_t* __restrict__ out_arg,
                  float* __restrict__ out_score) {
  // prop_scale and the entry's scores as [w - 1][s] (row pitch 32): every lane reads and writes its row position
  // unconditionally, the positions s > T - w are never read back
  __shared__ __align__(16) float s_sc[kTwo ? 2 : 1][32 * 32];
  __shared__ __align__(16) float s_curve[kNmsWarps][32 * 32];
  __shared__ int s_win[kNmsMaxP];              // window of proposal p: s | (s + w) << 8
  __shared__ int s_umax[33];                   // largest union u with fl(inter / u) > iou, per inter 0 .. 32 (0: none)
  const int n = blockIdx.x;
  const int v0 = vid_ptr[n], v1 = vid_ptr[n + 1];
  const int per = (v1 - v0 + (int)gridDim.y - 1) / (int)gridDim.y;
  const int c0 = v0 + (int)blockIdx.y * per, c1 = min(c0 + per, v1);
  if (c0 >= c1) return;
  const int P = T * (T + 1) / 2;
  for (int s = threadIdx.x; s < T; s += blockDim.x)
    for (int w = 1; s + w <= T; ++w) {
      const int p = prop_index(w, s, T);
      s_win[p] = s | ((s + w) << 8);
      s_sc[0][(w - 1) * 32 + s] = __ldg(scale0 + (int64_t)n * P + p);
      if (kTwo) s_sc[kTwo ? 1 : 0][(w - 1) * 32 + s] = __ldg(scale1 + (int64_t)n * P + p);
    }
  if (threadIdx.x <= 32) {
    const int i = threadIdx.x;
    int umax = 0;
    for (int u = i; u <= 64 && i > 0; ++u)
      if (__fdiv_rn((float)i, (float)u) > iou) umax = u;
    s_umax[i] = umax;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* cw = s_curve[warp];
  int win[kNmsSlots];
  uint32_t valid = 0;
#pragma unroll
  for (int k = 0; k < kNmsSlots; ++k) {
    const int p = 32 * k + lane;
    win[k] = p < P ? s_win[p] : (1 << 8);                          // past P: window (1, 0), never alive
    valid |= (p < P ? 1u : 0u) << k;
  }
  for (int e = c0 + warp; e < c1; e += kNmsWarps) {
    // ---- curve: lane = start s, window sums in clip order ----
    const float d0 = __ldg(dots0 + (int64_t)e * 32 + lane);
    const float d1 = kTwo ? __ldg(dots1 + (int64_t)e * 32 + lane) : 0.f;
    float r0 = 0.f, r1 = 0.f;
    __syncwarp();                                                   // the previous entry's reads of cw are done
#pragma unroll
    for (int w = 1; w <= 32; ++w) {
      const int src = (lane + w - 1) & 31;
      const float x0 = __shfl_sync(0xffffffffu, d0, src);
      r0 = (w == 1) ? x0 : __fadd_rn(r0, x0);
      const float s0 = __fmul_rn(r0, s_sc[0][(w - 1) * 32 + lane]);
      if (kTwo) {
        const float x1 = __shfl_sync(0xffffffffu, d1, src);
        r1 = (w == 1) ? x1 : __fadd_rn(r1, x1);
        const float s1 = __fmul_rn(r1, s_sc[kTwo ? 1 : 0][(w - 1) * 32 + lane]);
        cw[(w - 1) * 32 + lane] = __fadd_rn(__fmul_rn(w0, s0), __fmul_rn(w1, s1));
      } else {
        cw[(w - 1) * 32 + lane] = s0;
      }
    }
    __syncwarp();
    // ---- lane j: the windows p = 32 k + j ----
    float v[kNmsSlots];
#pragma unroll
    for (int k = 0; k < kNmsSlots; ++k) {
      const int s = win[k] & 0xff, en = win[k] >> 8;
      v[k] = cw[((en - s - 1) << 5) + s];
    }
    // ---- m rounds of greedy NMS; lane j keeps the pick of round j ----
    uint32_t alive = valid;
    int my_arg = -1;
    float my_score = -INFINITY;
    for (int j = 0; j < m; ++j) {
      float bv = -INFINITY;
      int bp = kNmsNone;
#pragma unroll
      for (int k = 0; k < kNmsSlots; ++k) {                         // p increases with k: strict > keeps the lower p
        const bool take = ((alive >> k) & 1u) && (bp == kNmsNone || v[k] > bv);
        bv = take ? v[k] : bv;
        bp = take ? 32 * k + lane : bp;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int op = __shfl_xor_sync(0xffffffffu, bp, o);
        const bool take = (op != kNmsNone) & ((bp == kNmsNone) | (ov > bv) | ((ov == bv) & (op < bp)));
        bv = take ? ov : bv;
        bp = take ? op : bp;
      }
      if (bp == kNmsNone) break;                                    // every window is suppressed: padding from here
      if (lane == j) { my_arg = bp; my_score = bv; }
      if (j + 1 == m) break;
      if (lane == (bp & 31)) alive &= ~(1u << (bp >> 5));            // the pick leaves the set even when iou >= 1
      const int pwin = s_win[bp];
      const int ps = pwin & 0xff, pe = pwin >> 8;
#pragma unroll
      for (int k = 0; k < kNmsSlots; ++k) {
        const int s = win[k] & 0xff, en = win[k] >> 8;
        const int inter = max(min(en, pe) - max(s, ps), 0);        // no overlap: s_umax[0] = 0 < any union
        alive &= ((en - s) + (pe - ps) - inter <= s_umax[inter]) ? ~(1u << k) : ~0u;
      }
    }
    if (lane < m) {
      const int64_t o = (int64_t)slot[e] * m + lane;
      out_arg[o] = my_arg;
      out_score[o] = my_score;
    }
  }
}

}  // namespace dkd

using namespace dkd;

extern "C" int dkd_moment_nms(const float* dots0, const float* scale0, const float* dots1, const float* scale1, float w0,
                              float w1, const int32_t* vid_ptr, const int32_t* slot, int32_t Nv, int32_t T, int32_t m,
                              float iou, int32_t* out_arg, float* out_score, void* stream) {
  if (!dots0 || !scale0 || !vid_ptr || !slot || !out_arg || !out_score || Nv < 0) return DKD_ERR_ARG;
  if ((dots1 == nullptr) != (scale1 == nullptr)) return DKD_ERR_ARG;
  if (!(iou >= 0.f)) return DKD_ERR_ARG;                            // negative or NaN
  if (T <= 0 || T > 32 || m < 1 || m > 16) return DKD_ERR_SHAPE;
  if (Nv == 0) return DKD_OK;
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // enough blocks for a few waves when the hits crowd into few videos; empty chunks return at once
  const int64_t want = ((int64_t)sms * 16 + Nv - 1) / Nv;
  dim3 grid(Nv, (unsigned)(want < 1 ? 1 : (want > 1024 ? 1024 : want)));
  if (dots1)
    moment_nms_kernel<true><<<grid, kNmsWarps * 32, 0, (cudaStream_t)stream>>>(dots0, scale0, dots1, scale1, w0, w1,
                                                                                vid_ptr, slot, T, m, iou, out_arg,
                                                                                out_score);
  else
    moment_nms_kernel<false><<<grid, kNmsWarps * 32, 0, (cudaStream_t)stream>>>(dots0, scale0, nullptr, nullptr, w0, w1,
                                                                                 vid_ptr, slot, T, m, iou, out_arg,
                                                                                 out_score);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}
