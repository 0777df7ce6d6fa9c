// Ranking kernels: warp-level streaming top-K selection, multi-shard merge, rank-of-GT,
// candidate CSR inversion and candidate sort.  Replace the host np.argsort of
// eval_q2m (method/eval.py:59-94): only the top-100 and the GT rank matter for R@K / medr / meanr.
//
// Order everywhere: score descending, video id ascending on equal scores — encoded as one
// 64-bit key (monotone float bits << 32 | ~id) so that "better" is a plain integer compare.
#include "dkd_common.cuh"

namespace dkd {

typedef unsigned long long u64;

// Bitonic sort (descending) of S (power of two) keys in shared memory by one warp.
__device__ __forceinline__ void warp_bitonic_desc(u64* a, int S, int lane) {
  for (int k = 2; k <= S; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < (S >> 1); t += 32) {
        // t-th compare-exchange pair of this stage
        const int i = ((t / j) * (j << 1)) + (t % j);
        const int l = i + j;
        const bool desc = ((i & k) == 0);
        const u64 x = a[i], y = a[l];
        const bool swap = desc ? (x < y) : (x > y);
        if (swap) { a[i] = y; a[l] = x; }
      }
      __syncwarp();
    }
  }
}

// Bitonic merge (descending) of a bitonic sequence of S keys by one warp.
__device__ __forceinline__ void warp_bitonic_merge_desc(u64* a, int S, int lane) {
  for (int j = S >> 1; j > 0; j >>= 1) {
    for (int t = lane; t < (S >> 1); t += 32) {
      const int i = ((t / j) * (j << 1)) + (t % j);
      const u64 x = a[i], y = a[i + j];
      if (x < y) { a[i] = y; a[i + j] = x; }
    }
    __syncwarp();
  }
}

// Streaming top-K by one warp: `list` = first H = S/2 slots (sorted desc, K <= H), queue = slots [H, S).
// flush: sort the queue alone, then keep the H best of (list, queue) with one compare-exchange pass against the
// reversed queue (the result is bitonic) and a bitonic merge — half the compare-exchanges of sorting all S slots.
struct WarpSelect {
  u64* buf;   // S slots
  int S, H, K, lane;
  int qn;     // queued (warp-uniform)
  u64 thresh; // K-th best so far (warp-uniform)
  __device__ void init(u64* b, int S_, int K_, int lane_) {
    buf = b; S = S_; H = S_ >> 1; K = K_; lane = lane_; qn = 0; thresh = 0ull;
    for (int i = lane; i < S; i += 32) buf[i] = 0ull;
    __syncwarp();
  }
  __device__ void flush() {
    warp_bitonic_desc(buf + H, H, lane);                 // queue, descending (empty slots are 0: they sink)
    for (int i = lane; i < H; i += 32) {                 // list[i] vs queue[H-1-i]: the H largest, bitonic
      const u64 x = buf[i], y = buf[S - 1 - i];
      if (y > x) buf[i] = y;
    }
    __syncwarp();
    warp_bitonic_merge_desc(buf, H, lane);
    for (int i = H + lane; i < S; i += 32) buf[i] = 0ull;
    __syncwarp();
    thresh = buf[K - 1];
    qn = 0;
  }
  // all 32 lanes call; `valid` lanes offer `key`
  __device__ void push(u64 key, bool valid) {
    const bool take = valid && key > thresh;
    const unsigned bal = __ballot_sync(0xffffffffu, take);
    if (bal == 0u) return;
    if (take) buf[H + qn + __popc(bal & ((1u << lane) - 1u))] = key;
    qn += __popc(bal);
    __syncwarp();
    if (qn + 32 > H) flush();
  }
};

// scores (M, Nv) dense, implicit ids id_base + n.
__global__ void topk_dense_kernel(const float* __restrict__ scores, int M, int Nv, int64_t ld, int K, int S,
                                  int id_base, float* __restrict__ out_scores, int32_t* __restrict__ out_ids) {
  extern __shared__ __align__(8) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  WarpSelect ws;
  ws.init(reinterpret_cast<u64*>(smem_raw) + (size_t)warp * S, S, K, lane);
  const float* row = scores + (int64_t)m * ld;
  for (int n0 = 0; n0 < Nv; n0 += 32) {
    const int n = n0 + lane;
    const bool valid = n < Nv;
    const float s = valid ? row[n] : 0.f;
    ws.push(pack_key(s, id_base + n), valid);
  }
  ws.flush();
  for (int j = lane; j < K; j += 32) {
    const u64 k = ws.buf[j];
    out_scores[(int64_t)m * K + j] = k ? key_score(k) : -INFINITY;
    out_ids[(int64_t)m * K + j] = k ? key_id(k) : -1;
  }
}

// Top-K SELECTION (unsorted) by a 4-pass radix select on the monotone 32-bit score key: one warp per row, a 256-bin
// histogram per pass in shared memory, then one compaction pass.  The candidate pass of engine.rank only needs the SET of
// the K best (they are rescored and sorted afterwards) and the K-th best approximate score (the certificate), so the
// streaming sort of topk_dense_kernel (7 bitonic flushes per row: ~30 k warp instructions) is not needed there.
// Order rule as everywhere: score descending, lower id first among equal scores (ties at the K-th score are taken in
// increasing column order until the quota is filled).
__global__ void __launch_bounds__(256)
select_topk_kernel(const float* __restrict__ scores, int M, int Nv, int64_t ld, int K, int id_base,
                   int32_t* __restrict__ out_ids, float* __restrict__ out_kth) {
  __shared__ int hist[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  const float* row = scores + (int64_t)m * ld;
  int32_t* oid = out_ids + (int64_t)m * K;
  if (Nv <= K) {                                            // everything is selected; pad the rest
    for (int n = lane; n < K; n += 32) oid[n] = n < Nv ? id_base + n : -1;
    if (lane == 0) out_kth[m] = -INFINITY;
    return;
  }
  int* h = hist[warp];
  uint32_t prefix = 0u;
  int need = K;                                             // rank of the wanted key among the keys matching `prefix`
#pragma unroll 1
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
#pragma unroll
    for (int i = 0; i < 8; ++i) h[lane * 8 + i] = 0;
    __syncwarp();
    for (int n = lane; n < Nv; n += 32) {
      const uint32_t key = float_key(row[n]);
      if (pass == 0 || ((key ^ prefix) >> (shift + 8)) == 0u) atomicAdd(&h[(key >> shift) & 255u], 1);
    }
    __syncwarp();
    // lane owns bins 8 lane .. 8 lane + 7; suffix sums from the top bin down
    int c[8], tot = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { c[i] = h[lane * 8 + i]; tot += c[i]; }
    int suf = tot;                                          // inclusive suffix sum over lanes >= this one
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_down_sync(0xffffffffu, suf, o);
      if (lane + o < 32) suf += v;
    }
    const bool mine = suf >= need && suf - tot < need;      // the wanted key falls into one of my bins
    int bin = 0, above = 0;
    if (mine) {
      int acc = suf - tot;                                  // keys in bins above mine
#pragma unroll
      for (int i = 7; i >= 0; --i) {
        if (acc + c[i] >= need) { bin = lane * 8 + i; above = acc; break; }
        acc += c[i];
      }
    }
    const unsigned who = __ballot_sync(0xffffffffu, mine);
    const int src = __ffs(who) - 1;
    bin = __shfl_sync(0xffffffffu, bin, src);
    above = __shfl_sync(0xffffffffu, above, src);
    prefix |= (uint32_t)bin << shift;
    need -= above;
    __syncwarp();
  }
  // prefix = key of the K-th best score; `need` of the keys equal to it are still wanted (first columns first)
  int cnt = 0, eq_taken = 0;
  for (int n0 = 0; n0 < Nv; n0 += 32) {
    const int n = n0 + lane;
    const uint32_t key = n < Nv ? float_key(row[n]) : 0u;
    const bool gt = n < Nv && key > prefix;
    const bool eq = n < Nv && key == prefix;
    const unsigned be = __ballot_sync(0xffffffffu, eq);
    const bool take = gt || (eq && eq_taken + __popc(be & ((1u << lane) - 1u)) < need);
    const unsigned bt = __ballot_sync(0xffffffffu, take);
    if (take) oid[cnt + __popc(bt & ((1u << lane) - 1u))] = id_base + n;
    cnt += __popc(bt);
    eq_taken += __popc(be);
  }
  if (lane == 0) out_kth[m] = key_float(prefix);
}

// Rank of `key` in buf[0, n) sorted descending, or -1 when it is not there.
__device__ __forceinline__ int find_key_desc(const u64* buf, int n, u64 key) {
  int lo = 0, hi = n;                                       // first position whose key is <= key
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (buf[mid] > key) lo = mid + 1; else hi = mid;
  }
  return (lo < n && buf[lo] == key) ? lo : -1;
}

// Payload move after a sort / merge: the input entry with key `key` copies its C payload words to the output rank its
// key landed on (if it survived).  Keys are unique per query, so every output rank receives one entry's words.
__device__ __forceinline__ void move_payload(const u64* buf, int n, u64 key, const uint32_t* __restrict__ src,
                                             uint32_t* __restrict__ dst_row, int C) {
  const int r = find_key_desc(buf, n, key);
  if (r < 0) return;
  for (int c = 0; c < C; ++c) dst_row[(int64_t)r * C + c] = src[c];
}

// (G, M, K) shard lists -> (M, K).  Entries with id < 0 are padding.  kPayload: also move the (G, M, K, C) payload
// words of every surviving entry to its output rank (out_payload (M, K, C); ranks without an entry are not written).
template <bool kPayload>
__global__ void merge_topk_kernel(const float* __restrict__ scores, const int32_t* __restrict__ ids, int G,
                                  int M, int K, int S, float* __restrict__ out_scores,
                                  int32_t* __restrict__ out_ids, const uint32_t* __restrict__ payload = nullptr,
                                  int C = 0, uint32_t* __restrict__ out_payload = nullptr) {
  extern __shared__ __align__(8) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  WarpSelect ws;
  ws.init(reinterpret_cast<u64*>(smem_raw) + (size_t)warp * S, S, K, lane);
  for (int g = 0; g < G; ++g) {
    const int64_t base = ((int64_t)g * M + m) * K;
    for (int j0 = 0; j0 < K; j0 += 32) {
      const int j = j0 + lane;
      bool valid = j < K;
      int id = valid ? ids[base + j] : -1;
      valid = valid && id >= 0;
      const float s = valid ? scores[base + j] : 0.f;
      ws.push(pack_key(s, id), valid);
    }
  }
  ws.flush();
  for (int j = lane; j < K; j += 32) {
    const u64 k = ws.buf[j];
    out_scores[(int64_t)m * K + j] = k ? key_score(k) : -INFINITY;
    out_ids[(int64_t)m * K + j] = k ? key_id(k) : -1;
  }
  if constexpr (kPayload) {
    for (int g = 0; g < G; ++g) {
      const int64_t base = ((int64_t)g * M + m) * K;
      for (int j = lane; j < K; j += 32) {
        const int id = ids[base + j];
        if (id >= 0)
          move_payload(ws.buf, K, pack_key(scores[base + j], id), payload + (base + j) * C,
                       out_payload + (int64_t)m * K * C, C);
      }
    }
  }
}

// Sort K candidates per query, keep K_out.  kPayload: also move the (M, K, C) payload words of every kept entry to its
// output rank (out_payload (M, K_out, C); ranks without an entry are not written).
template <bool kPayload>
__global__ void sort_candidates_kernel(const float* __restrict__ cs, const int32_t* __restrict__ cid, int M,
                                       int K, int K_out, int S, float* __restrict__ out_scores,
                                       int32_t* __restrict__ out_ids, const uint32_t* __restrict__ payload = nullptr,
                                       int C = 0, uint32_t* __restrict__ out_payload = nullptr) {
  extern __shared__ __align__(8) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  u64* buf = reinterpret_cast<u64*>(smem_raw) + (size_t)warp * S;
  for (int j = lane; j < S; j += 32) {
    u64 k = 0ull;
    if (j < K) {
      const int id = cid[(int64_t)m * K + j];
      if (id >= 0) k = pack_key(cs[(int64_t)m * K + j], id);
    }
    buf[j] = k;
  }
  __syncwarp();
  warp_bitonic_desc(buf, S, lane);
  for (int j = lane; j < K_out; j += 32) {
    const u64 k = buf[j];
    out_scores[(int64_t)m * K_out + j] = k ? key_score(k) : -INFINITY;
    out_ids[(int64_t)m * K_out + j] = k ? key_id(k) : -1;
  }
  if constexpr (kPayload) {
    for (int j = lane; j < K; j += 32) {
      const int64_t e = (int64_t)m * K + j;
      const int id = cid[e];
      if (id >= 0)
        move_payload(buf, K_out, pack_key(cs[e], id), payload + e * C, out_payload + (int64_t)m * K_out * C, C);
    }
  }
}

// rank of the best GT video: one warp per query.
__global__ void rank_of_gt_kernel(const float* __restrict__ scores, int M, int Nv, int64_t ld,
                                  const int32_t* __restrict__ gt_ptr, const int32_t* __restrict__ gt_ids,
                                  int32_t* __restrict__ out_rank) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const float* row = scores + (int64_t)m * ld;
  int best = Nv + 1;
  for (int g = gt_ptr[m]; g < gt_ptr[m + 1]; ++g) {
    const int gt = gt_ids[g];
    if (gt < 0 || gt >= Nv) continue;
    const float sg = row[gt];
    int cnt = 0;
    for (int n = lane; n < Nv; n += 32) {
      const float s = row[n];
      cnt += (s > sg) || (s == sg && n < gt);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    best = min(best, cnt + 1);
  }
  if (lane == 0) out_rank[m] = best;
}

__global__ void cand_hist_kernel(const int32_t* __restrict__ cand, int64_t total, int Nv, int id_base,
                                 int32_t* __restrict__ counts) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = cand[i] - id_base;
    if (n >= 0 && n < Nv) atomicAdd(&counts[n], 1);
  }
}
// single block exclusive scan: counts[0..Nv) -> vid_ptr[0..Nv]; counts reset to 0 (reused as cursors)
__global__ void cand_scan_kernel(int32_t* __restrict__ counts, int Nv, int32_t* __restrict__ vid_ptr) {
  __shared__ int part[1024];
  const int tid = threadIdx.x;
  const int per = (Nv + 1023) / 1024;
  const int b = tid * per, e = min(b + per, Nv);
  int s = 0;
  for (int i = b; i < e; ++i) s += counts[i];
  part[tid] = s;
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int i = 0; i < 1024; ++i) { int t = part[i]; part[i] = run; run += t; }
    vid_ptr[Nv] = run;
  }
  __syncthreads();
  int run = part[tid];
  for (int i = b; i < e; ++i) {
    const int c = counts[i];
    vid_ptr[i] = run;
    run += c;
    counts[i] = 0;
  }
}
__global__ void cand_fill_kernel(const int32_t* __restrict__ cand, int64_t total, int K, int Nv, int id_base,
                                 int32_t* __restrict__ cursors, const int32_t* __restrict__ vid_ptr,
                                 int32_t* __restrict__ q_list, int32_t* __restrict__ slot) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = cand[i] - id_base;
    if (n >= 0 && n < Nv) {
      const int e = vid_ptr[n] + atomicAdd(&cursors[n], 1);
      q_list[e] = (int)(i / K);
      slot[e] = (int)i;
    }
  }
}

// ---- ambiguous-pair selection: pairs (m, n) whose bf16 argmax gap is below tau ------------------
__global__ void pair_hist_kernel(const float* __restrict__ gap, int M, int Nv, int64_t ld, float tau,
                                 int32_t* __restrict__ counts) {
  const int64_t total = (int64_t)M * Nv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int m = (int)(i / Nv), n = (int)(i % Nv);
    if (gap[(int64_t)m * ld + n] < tau) atomicAdd(&counts[n], 1);
  }
}
__global__ void pair_fill_kernel(const float* __restrict__ gap, int M, int Nv, int64_t ld, float tau,
                                 int32_t* __restrict__ cursors, const int32_t* __restrict__ vid_ptr,
                                 int32_t* __restrict__ q_list, int32_t* __restrict__ slot, int64_t cap) {
  const int64_t total = (int64_t)M * Nv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int m = (int)(i / Nv), n = (int)(i % Nv);
    if (gap[(int64_t)m * ld + n] < tau) {
      const int64_t e = (int64_t)vid_ptr[n] + atomicAdd(&cursors[n], 1);
      if (e < cap) { q_list[e] = m; slot[e] = (int)((int64_t)m * ld + n); }
    }
  }
}
// ---- flagged-pair lists from the GEMM's bit matrix: one block per 32 videos (one word column) ----------------
// flags (M, W) uint32, bit (n & 31) of word [m][n >> 5].  Per video a contiguous run of q_list / slot entries
// (any order inside the run), runs placed by a global cursor: vid_begin[n], vid_cnt[n].
__global__ void __launch_bounds__(256)
flag_select_kernel(const uint32_t* __restrict__ flags, int M, int Nv, int W, int64_t ld, int32_t* __restrict__ cursor,
                   int32_t* __restrict__ vid_begin, int32_t* __restrict__ vid_cnt, int32_t* __restrict__ q_list,
                   int32_t* __restrict__ slot, int64_t cap) {
  __shared__ int cnt[32], base[32], cur[32];
  const int g = blockIdx.x, tid = threadIdx.x;
  if (tid < 32) { cnt[tid] = 0; cur[tid] = 0; }
  __syncthreads();
  for (int m = tid; m < M; m += 256) {
    uint32_t w = flags[(int64_t)m * W + g];
    while (w) { const int b = __ffs(w) - 1; w &= w - 1; atomicAdd(&cnt[b], 1); }
  }
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int b = 0; b < 32; ++b) { base[b] = tot; tot += cnt[b]; }
    const int start = atomicAdd(cursor, tot);
    for (int b = 0; b < 32; ++b) base[b] += start;
  }
  __syncthreads();
  if (tid < 32 && g * 32 + tid < Nv) { vid_begin[g * 32 + tid] = base[tid]; vid_cnt[g * 32 + tid] = cnt[tid]; }
  for (int m = tid; m < M; m += 256) {
    uint32_t w = flags[(int64_t)m * W + g];
    while (w) {
      const int b = __ffs(w) - 1; w &= w - 1;
      const int64_t e = (int64_t)base[b] + atomicAdd(&cur[b], 1);
      if (e < cap) { q_list[e] = m; slot[e] = (int)((int64_t)m * ld + g * 32 + b); }
    }
  }
}

// out[slot[e]] = fl(wa * a[e]) + fl(wb * b[e])  (b may be null: out[slot[e]] = a[e])
// kDetail: also payload[slot[e]][0, 1] = (arg_a[e], bits of a[e]) and, with b, [2, 3] = (arg_b[e], bits of b[e]).
template <bool kDetail>
__global__ void scatter_fuse_kernel(const float* __restrict__ a, const float* __restrict__ b, float wa, float wb,
                                    const int32_t* __restrict__ slot, const int32_t* __restrict__ total_ptr,
                                    float* __restrict__ out, const int32_t* __restrict__ arg_a = nullptr,
                                    const int32_t* __restrict__ arg_b = nullptr, uint32_t* __restrict__ payload = nullptr,
                                    int C = 0) {
  const int64_t total = *total_ptr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = b ? __fadd_rn(__fmul_rn(wa, a[i]), __fmul_rn(wb, b[i])) : a[i];
    out[slot[i]] = v;
    if constexpr (kDetail) {
      uint32_t* pd = payload + (int64_t)slot[i] * C;
      pd[0] = (uint32_t)arg_a[i];
      pd[1] = __float_as_uint(a[i]);
      if (b) {
        pd[2] = (uint32_t)arg_b[i];
        pd[3] = __float_as_uint(b[i]);
      }
    }
  }
}

}  // namespace dkd

using namespace dkd;

static int pow2_at_least(int v) {
  int p = 32;
  while (p < v) p <<= 1;
  return p;
}

extern "C" int dkd_topk(const float* scores, int32_t M, int32_t Nv, int64_t ld, int32_t K, int32_t id_base,
                        float* out_scores, int32_t* out_ids, void* stream) {
  if (!scores || !out_scores || !out_ids || M < 0 || Nv < 0 || ld < Nv) return DKD_ERR_ARG;
  if (K <= 0 || K > 256) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  const int S = 2 * pow2_at_least(K);
  const int wpb = 4;
  const size_t smem = (size_t)wpb * S * sizeof(u64);
  topk_dense_kernel<<<(M + wpb - 1) / wpb, wpb * 32, smem, (cudaStream_t)stream>>>(
      scores, M, Nv, ld, K, S, id_base, out_scores, out_ids);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_select_topk(const float* scores, int32_t M, int32_t Nv, int64_t ld, int32_t K, int32_t id_base,
                               int32_t* out_ids, float* out_kth, void* stream) {
  if (!scores || !out_ids || !out_kth || M < 0 || Nv < 0 || ld < Nv) return DKD_ERR_ARG;
  if (K <= 0) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  select_topk_kernel<<<(M + 7) / 8, 256, 0, (cudaStream_t)stream>>>(scores, M, Nv, ld, K, id_base, out_ids, out_kth);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_merge_topk(const float* scores, const int32_t* ids, int32_t G, int32_t M, int32_t K,
                              float* out_scores, int32_t* out_ids, void* stream) {
  if (!scores || !ids || !out_scores || !out_ids || G <= 0 || M < 0) return DKD_ERR_ARG;
  if (K <= 0 || K > 256) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  const int S = 2 * pow2_at_least(K);
  const int wpb = 4;
  const size_t smem = (size_t)wpb * S * sizeof(u64);
  merge_topk_kernel<false><<<(M + wpb - 1) / wpb, wpb * 32, smem, (cudaStream_t)stream>>>(scores, ids, G, M, K, S,
                                                                                        out_scores, out_ids);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_sort_candidates(const float* cand_scores, const int32_t* cand_ids, int32_t M, int32_t K,
                                   int32_t K_out, float* out_scores, int32_t* out_ids, void* stream) {
  if (!cand_scores || !cand_ids || !out_scores || !out_ids || M < 0) return DKD_ERR_ARG;
  if (K <= 0 || K > 512 || K_out <= 0 || K_out > K) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  const int S = pow2_at_least(K);
  const int wpb = 4;
  const size_t smem = (size_t)wpb * S * sizeof(u64);
  sort_candidates_kernel<false><<<(M + wpb - 1) / wpb, wpb * 32, smem, (cudaStream_t)stream>>>(
      cand_scores, cand_ids, M, K, K_out, S, out_scores, out_ids);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_merge_topk_payload(const float* scores, const int32_t* ids, const uint32_t* payload, int32_t G,
                                      int32_t M, int32_t K, int32_t C, float* out_scores, int32_t* out_ids,
                                      uint32_t* out_payload, void* stream) {
  if (!scores || !ids || !payload || !out_scores || !out_ids || !out_payload || G <= 0 || M < 0) return DKD_ERR_ARG;
  if (K <= 0 || K > 256 || C <= 0 || C > 8) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  const int S = 2 * pow2_at_least(K);
  const int wpb = 4;
  const size_t smem = (size_t)wpb * S * sizeof(u64);
  merge_topk_kernel<true><<<(M + wpb - 1) / wpb, wpb * 32, smem, (cudaStream_t)stream>>>(
      scores, ids, G, M, K, S, out_scores, out_ids, payload, C, out_payload);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_sort_candidates_payload(const float* cand_scores, const int32_t* cand_ids, const uint32_t* payload,
                                           int32_t M, int32_t K, int32_t K_out, int32_t C, float* out_scores,
                                           int32_t* out_ids, uint32_t* out_payload, void* stream) {
  if (!cand_scores || !cand_ids || !payload || !out_scores || !out_ids || !out_payload || M < 0) return DKD_ERR_ARG;
  if (K <= 0 || K > 512 || K_out <= 0 || K_out > K || C <= 0 || C > 8) return DKD_ERR_SHAPE;
  if (M == 0) return DKD_OK;
  const int S = pow2_at_least(K);
  const int wpb = 4;
  const size_t smem = (size_t)wpb * S * sizeof(u64);
  sort_candidates_kernel<true><<<(M + wpb - 1) / wpb, wpb * 32, smem, (cudaStream_t)stream>>>(
      cand_scores, cand_ids, M, K, K_out, S, out_scores, out_ids, payload, C, out_payload);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_rank_of_gt(const float* scores, int32_t M, int32_t Nv, int64_t ld, const int32_t* gt_ptr,
                              const int32_t* gt_ids, int32_t* out_rank, void* stream) {
  if (!scores || !gt_ptr || !gt_ids || !out_rank || M < 0 || Nv < 0 || ld < Nv) return DKD_ERR_ARG;
  if (M == 0) return DKD_OK;
  const int wpb = 8;
  rank_of_gt_kernel<<<(M + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(scores, M, Nv, ld, gt_ptr,
                                                                              gt_ids, out_rank);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_candidates_to_csr(const int32_t* cand_ids, int32_t M, int32_t K, int32_t Nv,
                                     int32_t id_base, int32_t* counts, int32_t* vid_ptr, int32_t* q_list,
                                     int32_t* slot, void* stream) {
  if (!cand_ids || !counts || !vid_ptr || !q_list || !slot || M < 0 || K <= 0 || Nv <= 0) return DKD_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = (int64_t)M * K;
  DKD_CUDA_TRY(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)Nv, st));
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  cand_hist_kernel<<<(unsigned)blocks, 256, 0, st>>>(cand_ids, total, Nv, id_base, counts);
  DKD_LAUNCH_CHECK();
  cand_scan_kernel<<<1, 1024, 0, st>>>(counts, Nv, vid_ptr);
  DKD_LAUNCH_CHECK();
  cand_fill_kernel<<<(unsigned)blocks, 256, 0, st>>>(cand_ids, total, K, Nv, id_base, counts, vid_ptr, q_list, slot);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_scatter_fuse(const float* a, const float* b, float wa, float wb, const int32_t* slot,
                                const int32_t* vid_ptr, int32_t Nv, int64_t max_entries, float* out, void* stream) {
  if (!a || !slot || !vid_ptr || !out || Nv <= 0 || max_entries < 0) return DKD_ERR_ARG;
  if (max_entries == 0) return DKD_OK;
  int64_t blocks = (max_entries + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  scatter_fuse_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, b, wa, wb, slot, vid_ptr + Nv, out);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_scatter_fuse_detail(const float* a, const float* b, float wa, float wb, const int32_t* arg_a,
                                       const int32_t* arg_b, const int32_t* slot, const int32_t* vid_ptr, int32_t Nv,
                                       int64_t max_entries, float* out, uint32_t* payload, int32_t C, void* stream) {
  if (!a || !arg_a || !slot || !vid_ptr || !out || !payload || Nv <= 0 || max_entries < 0) return DKD_ERR_ARG;
  if ((b == nullptr) != (arg_b == nullptr)) return DKD_ERR_ARG;
  if (C < (b ? 4 : 2)) return DKD_ERR_SHAPE;
  if (max_entries == 0) return DKD_OK;
  int64_t blocks = (max_entries + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  scatter_fuse_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, b, wa, wb, slot, vid_ptr + Nv, out,
                                                                                arg_a, arg_b, payload, C);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_select_pairs_csr(const float* gap, int32_t M, int32_t Nv, int64_t ld, float tau, int64_t cap,
                                    int32_t* counts, int32_t* vid_ptr, int32_t* q_list, int32_t* slot,
                                    void* stream) {
  if (!gap || !counts || !vid_ptr || !q_list || !slot || M < 0 || Nv <= 0 || ld < Nv || cap < 0) return DKD_ERR_ARG;
  if ((int64_t)M * ld > 0x7fffffffLL) return DKD_ERR_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  DKD_CUDA_TRY(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)Nv, st));
  const int blocks = 148 * 8;
  pair_hist_kernel<<<blocks, 256, 0, st>>>(gap, M, Nv, ld, tau, counts);
  DKD_LAUNCH_CHECK();
  cand_scan_kernel<<<1, 1024, 0, st>>>(counts, Nv, vid_ptr);
  DKD_LAUNCH_CHECK();
  pair_fill_kernel<<<blocks, 256, 0, st>>>(gap, M, Nv, ld, tau, counts, vid_ptr, q_list, slot, cap);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_select_flagged(const uint32_t* flags, int32_t M, int32_t Nv, int64_t ld, int64_t cap,
                                  int32_t* cursor, int32_t* vid_begin, int32_t* vid_cnt, int32_t* q_list,
                                  int32_t* slot, void* stream) {
  if (!flags || !cursor || !vid_begin || !vid_cnt || !q_list || !slot || M < 0 || Nv <= 0 || ld < Nv || cap < 0)
    return DKD_ERR_ARG;
  if ((int64_t)M * ld > 0x7fffffffLL) return DKD_ERR_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  DKD_CUDA_TRY(cudaMemsetAsync(cursor, 0, sizeof(int32_t), st));
  const int W = (Nv + 31) / 32;
  flag_select_kernel<<<W, 256, 0, st>>>(flags, M, Nv, W, ld, cursor, vid_begin, vid_cnt, q_list, slot, cap);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}
