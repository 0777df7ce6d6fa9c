// Exact (fp32-grade) clip-scale scores on the tcgen05 tensor cores.
//
//   d[i]        = qn[m] . clips[n, i]                       i = 0..T-1      tcgen05.mma kind::tf32, 3 products
//   S[p(w, s)]  = (d[s] + d[s+1] + ... + d[s+w-1]) * prop_scale[n, p]       fp32 running sums in registers
//   out_max     = max_p S,   out_arg = first argmax_p       (torch.max tie rule)
//
// fp32 accuracy from tf32 tensor cores by operand splitting: x = hi + lo with hi = tf32(x), lo = tf32(x - hi)
// (done by the staging warps on the way into shared memory), d = lo.hi + hi.lo + hi.hi accumulated in one fp32 TMEM
// accumulator — relative error per product ~2^-21, inside the summation-order noise of an fp32 einsum.
// This is the fp32 flavour of get_clip_scale_scores (SURVEY §8 N3): (a) the exact drop-in path (dense),
// (b) re-resolution of the pairs whose bf16 argmax is ambiguous, (c) rescoring of the top-K candidates;
// (b) and (c) address the pairs through a CSR by video (vid_ptr / q_list).
//
// One persistent CTA per SM walks videos; a tile = 128 list entries of one video (UMMA M = 128, N = 32 clips).
// The A operand (query rows) lives in TENSOR MEMORY: with N = 32 an MMA that re-reads a 128-row A tile from
// shared memory is shared-memory-bandwidth bound (5 KB per 16-cycle MMA), from TMEM it runs at the MMA floor.
//   warps 0-3   scan: tcgen05.ld of the lane's 32 dots, 528 running window sums x scale, max/first argmax
//               (thread = tile row; 8 independent running maxima per thread)
//   warps 4-11  stagers (two per TMEM lane quarter, alternating K blocks): cp.async gather of the fp32 query rows
//               (32 features per K block) into a per-warp ring, split into tf32 hi / lo, tcgen05.st.16x256b into
//               the A ring (64 columns per stage)
//   warp 12     tcgen05.mma issuer (one elected lane, A from TMEM, B from smem) + TMEM allocation
//               (512 columns: 2 x 32 accumulator + 7 x 64 A ring)
//   warp 13     B loader: one cp.async.bulk per video of its pre-packed clip planes (dkd_pack_clips_tf32: the
//               shared-memory image of the B operand — tf32 hi / lo planes, K-major SWIZZLE_128B)
#include "dkd_umma.cuh"
#include "dkd_scan.cuh"

namespace dkd {

constexpr int kXRows = 128;                 // list entries per tile
constexpr int kXKB = 32;                    // fp32 features per K block (one 128-byte swizzle row)
constexpr int kXScanWarps = 4;              // one per TMEM lane quarter: thread = tile row
constexpr int kXStageWarps = 8;             // two per TMEM lane quarter, alternating K blocks
constexpr int kXStagers = 4 * 32;            // stager threads that fill one A stage (one warp per quarter)
constexpr int kXMmaWarp = kXScanWarps + kXStageWarps;
constexpr int kXLoadWarp = kXMmaWarp + 1;   // B-operand loader (cp.async.bulk of the pre-packed clip planes)
constexpr int kXThreads = (kXLoadWarp + 1) * 32;
constexpr int kXMaxAStages = 7;             // A ring stages in TMEM: (512 - 2 x accumulator width) / 64
constexpr int kXBStages = 3;                // rows mode: B ring stages in shared memory
constexpr uint32_t kXBPlane = 32 * 128;      // 4 KB : 32 clips x 128 B
constexpr int kXTmemCols = 512;
constexpr uint32_t kXRowPitch = 128;        // staged fp32 row of one K block; 16-byte chunk c of row r sits at
                                            // chunk c ^ ((r & 1) << 2): conflict-free cp.async writes and LDS.128 reads
constexpr uint32_t kXSlotBytes = 32 * kXRowPitch;
constexpr uint32_t kXScanScratch = 32 * kXRows * 4;   // 16 KB per scan group: the tile's dots, [clip][row]
// per-stager-warp cp.async ring: kRing slots (kRing - 1 of the warp's K blocks in flight), 3 normally, 2 when D > 448

struct ExactParams {
  const float* q; int M;
  const float* planes; const float* scale;
  int Nv, T, D;
  int b_bufs;
  int R, Npad;                 // rows mode: rows per video, padded to a multiple of 16 (UMMA N)
  const uint8_t* mask;         // rows mode: (Nv, R) or null
  float* out_max; int32_t* out_arg; int64_t ld_out;
  const int32_t* vid_ptr; const int32_t* vid_cnt; const int32_t* q_list; const int32_t* out_slot;
  unsigned wait_ns;            // sleep between mbarrier polls of the non-critical warps (0: spin)
  // mode 2 (dense clip windows, kXGroup videos per tile): Nv = number of WORK ITEMS = video groups x tile chunks
  int Nv_real, tile_chunks, tiles_per_chunk;
  // mode 4 (linear layer: out = act(x_hat . W^T + bias)): "videos" are 128-row tiles of the packed weight matrix,
  // work items = (row chunk, weight tile) with the weight tile fastest (CTAs running together share the rows of x in L2)
  int64_t list_stride;         // > 0: no vid_ptr — video n's entries are q_list[n * list_stride ...), vid_cnt[n] of them,
                               // and results are scattered to the dense matrix at (query, video)
  const int32_t* known_key;    // mode 0, optional: dense (M, known_ld) key clips to confirm (dkd_scan.cuh window_scan_known)
  int64_t known_ld;
  const float2* row_ss;        // optional per-row (scale, shift): x_hat = x * scale + shift (LayerNorm prologue)
  const float* bias;           // optional (n_cols)
  int relu, n_cols;
};
constexpr int kXGroup = 4;                   // mode 2: videos sharing one staged A tile (UMMA N = 4 x 32 clips)
// Which window scan runs (dkd_scan.cuh).  In isolation (tools/micro/scan2_micro.cu, profiles/r2_scan_micro.md) the
// two-phase scan needs 5.2 k cycles per warp-scan against 7.4 k for v1 and the known-key confirmation 3.2-3.4 k; inside
// this kernel the list forms are bound by the query-row gather of the stagers, so the whole-step A/B
// (profiles/r2_ab_exact_scan.md) separates the variants by 0.1-0.4 ms only: v1 for the full scan + scalar known-key
// confirmation for the candidate pass measured best and is the default.  The dense form (mode 2) keeps v1: with two
// scan warps per scheduler it is pipe bound and the two-phase scan gains nothing.
#ifndef DKD_X_LIST_SCAN
#define DKD_X_LIST_SCAN 0      // full scan of the list form: 0 = v1, 1 = two-phase scalar, 2 = two-phase packed
#endif
#ifndef DKD_X_KNOWN
#define DKD_X_KNOWN 1          // known-key confirmation: 0 = off (full scan), 1 = scalar phase 1, 2 = packed phase 1
#endif
#ifndef DKD_X_STREAM_B0
#define DKD_X_STREAM_B0 0      // 1: mode 0 streams the video's clip planes per K block (like mode 1) instead of keeping them
                               // resident, which frees 72 KB of shared memory for a deeper stager ring (DKD_X_RING0).
                               // MEASURED (round 2, whole step, same box): exact kernel's four calls 3.15 ms (ring 5) /
                               // 2.96 ms (ring 4) against 2.93 ms resident with ring 3 — more query rows in flight do
                               // not help: the list forms are bound by the stagers' instruction stream, not by latency
#endif
#ifndef DKD_X_RING0
#define DKD_X_RING0 5          // stager ring slots of mode 0 when B is streamed (ring - 1 query-row blocks in flight per warp)
#endif
constexpr bool kXStreamB0 = DKD_X_STREAM_B0 != 0;
constexpr int kXListScan = DKD_X_LIST_SCAN;
constexpr int kXKnown = DKD_X_KNOWN;
constexpr bool kXTwoPhaseList = kXListScan != 0 || kXKnown != 0;   // the scan scratch in shared memory is needed

struct __align__(8) ExactCtl {
  uint64_t a_full[kXMaxAStages], a_empty[kXMaxAStages];
  uint64_t b_full[kXBStages], b_empty[kXBStages];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// hi = tf32(x) rounded to nearest (ties away from zero: add half an ulp to the magnitude bits, clear the low 13
// bits — cvt.rna.tf32.f32 without its inf/nan handling; operands are finite L2-normalised features);
// lo = x - hi exactly (<= 13 significant bits).  The tensor core reads only the tf32 part of lo (drops its low
// 13 bits: <= 2^-21 |x|, sign-symmetric because hi is rounded to nearest).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// 16 lanes x 32 columns: reg 4j+e -> (lane g = tid/4, col 8j + 2(tid%4) + e), reg 4j+2+e -> lane g + 8
// (layout verified on hardware: tools/micro/tmem_layout.cu)
__device__ __forceinline__ void tmem_st_16x256b_x4(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.16x256b.x4.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem], tf32 x tf32 -> fp32
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// kind::tf32: D = f32, A = B = tf32 (format 2), both K-major
__host__ __device__ __forceinline__ uint32_t make_idesc_tf32(int n, int m) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// byte offset of 16-byte chunk c (0..7) of row r inside a K-major SWIZZLE_128B plane (8-row groups of 1024 B)
__device__ __forceinline__ uint32_t sw128_off(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}

__device__ __forceinline__ void video_range(const ExactParams& p, int n, int& e0, int& count) {
  if (p.vid_ptr) { e0 = p.vid_ptr[n]; count = p.vid_cnt ? p.vid_cnt[n] : p.vid_ptr[n + 1] - e0; }
  else if (p.list_stride > 0) {
    e0 = (int)((int64_t)n * p.list_stride);
    count = p.vid_cnt[n];
    if (count > (int)p.list_stride) count = (int)p.list_stride;
  }
  else { e0 = 0; count = p.M; }
}

// mode 2 work item -> (video group, first query row, number of query rows)
__device__ __forceinline__ void item_range(const ExactParams& p, int item, int& group, int& row0, int& count) {
  group = item / p.tile_chunks;
  const int chunk = item - group * p.tile_chunks;
  row0 = chunk * p.tiles_per_chunk * kXRows;
  const int rows = p.tiles_per_chunk * kXRows;
  count = p.M - row0 < rows ? p.M - row0 : rows;
}

// mode 4 work item -> (weight tile, first row, number of rows): weight tile fastest
__device__ __forceinline__ void item_range_linear(const ExactParams& p, int item, int& wtile, int& row0, int& count) {
  wtile = item % p.Nv_real;
  const int chunk = item / p.Nv_real;
  row0 = chunk * p.tiles_per_chunk * kXRows;
  const int rows = p.tiles_per_chunk * kXRows;
  count = p.M - row0 < rows ? p.M - row0 : rows;
}

// kMode 0: clip windows (B = the video's 32 clips, resident; scan = T(T+1)/2 window cosines).
// kMode 1: rows max (B = the video's R <= 128 rows, streamed per K block through a ring; scan = masked max).
// kMode 2: clip windows, DENSE only.  Measurements (tools/micro/scan_micro.cu, DESIGN.md): one window scan is a
//          latency-bound instruction stream (7.4 k cycles per 32 rows in isolation, ~9.9 k next to the stagers) and it
//          paces the whole kernel; two independent scans per scheduler overlap perfectly.  So mode 2 runs TWO scan
//          groups (warps 0-3 take the even tiles = accumulator buffer 0, warps 8-11 the odd tiles = buffer 1) and
//          pays for the second group with stager warps: kXGroup = 4 videos share every staged A tile (their clip planes
//          form one N = 128 B operand, streamed per K block like mode 1), which cuts the staging work per pair 4 x, so
//          one stager warp per TMEM lane quarter (warps 4-7) is enough.  Same 14 warps, same 128 registers per thread.
//          Modes 0 / 1 keep one scan group and two stager sets (list forms: every video has its own query list).
// kMode 4: linear layer on the same pipeline as mode 1 (fp32-grade tf32 x 3): A = rows of x (optionally normalised on
//          the fly by a per-row scale / shift: the LayerNorm in front of the projection), B = a 128-row tile of the
//          pre-packed weight matrix streamed per K block, epilogue = + bias, optional ReLU, fp32 store of the tile.
// kDots (mode 0, CSR list form): the scan warps store each entry's 32 dots to p.out_max + 32 * entry instead of
//          scanning (dkd_clip_dots_list); prop_scale is not read.
template <int kMode, bool kT32, int kXRing, bool kDots = false>
__global__ void __launch_bounds__(kXThreads, 1)
exact_umma_kernel(const ExactParams p) {
  constexpr int kDW = kMode == 0 ? 32 : 128;                    // accumulator columns per TMEM buffer
  constexpr int kScaleBufs = kMode == 2 ? kXGroup : 2;
  constexpr int kStageSets = kMode == 2 ? 1 : 2;                // stager warps per TMEM lane quarter
  constexpr int kScanGroups = (kMode == 0 && kXTwoPhaseList) ? 1 : 0;   // scan scratch (two-phase / known-key scans)
  constexpr bool kResB = kMode == 0 && !kXStreamB0;             // B operand resident per video (else streamed per K block)
  constexpr uint32_t kXACol0 = 2 * kDW;                         // first A-ring column
  constexpr int kXStages = (kXTmemCols - 2 * kDW) / 64;         // A ring stages: 7 / 4
  extern __shared__ __align__(1024) uint8_t smem_raw_x[];
  __shared__ __align__(16) float s_scale[kScaleBufs][32 * 32];   // prop_scale of the current video(s) as [w - 1][s]
                                                        // (scan warps; mode 0: double buffered): 16-byte loads at
                                                        // compile-time offsets
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw_x) + 1023) & ~(uintptr_t)1023);
  const int num_kb = p.D / kXKB;
  // mode 0: [buf][kb][plane] x 4 KB, one buffer per video; mode 1: [stage][plane] x Npad x 128 B, one stage per K block
  const uint32_t b_buf_bytes = kResB ? (uint32_t)num_kb * 2u * kXBPlane : 2u * (uint32_t)p.Npad * 128u;
  uint8_t* sB = smem;
  uint8_t* sS = sB + (size_t)(kResB ? p.b_bufs : kXBStages) * b_buf_bytes;   // [stager warp][slot][32 rows] x 128 B
  // scan scratch (clip-window modes): per scan group 32 x 128 floats, column = tile row (two-phase scan, dkd_scan.cuh)
  float* sD = reinterpret_cast<float*>(sS + (size_t)(4 * kStageSets) * kXRing * kXSlotBytes);
  ExactCtl* ctl = reinterpret_cast<ExactCtl*>(reinterpret_cast<uint8_t*>(sD) + (size_t)kScanGroups * kXScanScratch);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t b_bufs = (uint32_t)p.b_bufs;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kXStages; ++i) { mbar_init(&ctl->a_full[i], kXStagers); mbar_init(&ctl->a_empty[i], 1); }
    for (int i = 0; i < kXBStages; ++i) { mbar_init(&ctl->b_full[i], 1); mbar_init(&ctl->b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&ctl->tmem_full[i], 1);
      mbar_init(&ctl->tmem_empty[i], kXScanWarps);
    }
    fence_barrier_init();
  }
  if (warp == kXMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctl->tmem_base)), "n"(kXTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = ctl->tmem_base;

  if (warp >= kXScanWarps && warp < kXScanWarps + 4 * kStageSets) {
    // ===================== stagers =====================
    // Query rows are gathered as fp32 (coalesced 128-byte row segments) by cp.async into a private per-warp
    // ring (kXRing - 1 K blocks in flight per warp: the gather is latency bound, the bytes in flight set its
    // bandwidth), read back as tcgen05.st.16x256b fragments, split into tf32 hi / lo and stored to the TMEM A
    // ring, whose 7 stages decouple the stagers from the MMA.
    const int quarter = warp & 3, par = (warp - kXScanWarps) >> 2;   // this warp stages items j = par (mod kStageSets)
    const int g = lane >> 2, t = lane & 3;
    const int cl_row = lane >> 3, cl_chunk = lane & 7;          // cp.async: 4 rows x 8 chunks per instruction
    const uint32_t a_lane = tmem_base + ((uint32_t)(quarter * 32) << 16) + kXACol0;
    const int sw = warp - kXScanWarps;                          // 0..7
    const uint32_t ring0 = smem_u32(sS) + (uint32_t)sw * kXRing * kXSlotBytes;
    const uint8_t* ring_ptr = sS + (size_t)sw * kXRing * kXSlotBytes;
    uint32_t it_base = 0;                                       // A ring counter of item 0 of the current video
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int e0, count, row_base = 0;
      if (kMode == 2) { int g_; item_range(p, n, g_, row_base, count); e0 = 0; }
      else if (kMode == 4) { int g_; item_range_linear(p, n, g_, row_base, count); e0 = 0; }
      else video_range(p, n, e0, count);
      if (count <= 0) continue;
      int ss_tile = -1;                                         // mode 4: tile whose row scale / shift is cached
      float2 ss[4];
      const int nitems = ((count + kXRows - 1) / kXRows) * num_kb;
      // item j = (tile j / num_kb, K block j % num_kb) of this video
      int t_cached = -1;
      const float* src_cached[8];
      uint32_t live_mask = 0;
      int iss_tile = 0, iss_kb = par;                           // (tile, K block) of this warp's next item to issue
      while (iss_kb >= num_kb) { iss_kb -= num_kb; ++iss_tile; }
      auto issue = [&](int slot) {
        const int tile = iss_tile, kb = iss_kb;
        iss_kb += kStageSets;
        while (iss_kb >= num_kb) { iss_kb -= num_kb; ++iss_tile; }
        if (tile != t_cached) {
          t_cached = tile;
          live_mask = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = tile * kXRows + quarter * 32 + 4 * i + cl_row;
            const bool live = r < count;
            const int64_t qrow = live ? (p.q_list ? (int64_t)p.q_list[e0 + r] : (int64_t)(row_base + r)) : 0;
            src_cached[i] = p.q + qrow * p.D + 4 * cl_chunk;
            live_mask |= (live ? 1u : 0u) << i;
          }
        }
        // rows 4i + cl_row: (row & 1) == (cl_row & 1)
        const uint32_t dst = ring0 + (uint32_t)slot * kXSlotBytes + (uint32_t)cl_row * kXRowPitch +
                             (uint32_t)((cl_chunk ^ ((cl_row & 1) << 2)) << 4);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          cp_async16(dst + (uint32_t)(4 * i) * kXRowPitch, src_cached[i] + kb * kXKB, ((live_mask >> i) & 1u) ? 16u : 0u);
      };
      auto store = [&](int j, int slot_i) {
        // fragments of item j: rows 16h + g + 8u ((row & 1) == (g & 1)), features 16c + 4t .. +3 (chunk 4c + t)
        const uint8_t* slot = ring_ptr + (size_t)slot_i * kXSlotBytes;
        float4 v[8];
#pragma unroll
        for (int hu = 0; hu < 4; ++hu)
#pragma unroll
          for (int c = 0; c < 2; ++c)
            v[2 * hu + c] = *reinterpret_cast<const float4*>(
                slot + (16 * (hu >> 1) + g + 8 * (hu & 1)) * kXRowPitch + (((4 * c + t) ^ ((g & 1) << 2)) << 4));
        if (kMode == 4) {
          if (p.row_ss) {                                       // x_hat = x * scale + shift of the row (LayerNorm prologue)
            const int tile_j = j / num_kb;
            if (tile_j != ss_tile) {
              ss_tile = tile_j;
#pragma unroll
              for (int hu = 0; hu < 4; ++hu) {
                const int r = tile_j * kXRows + quarter * 32 + 16 * (hu >> 1) + g + 8 * (hu & 1);
                ss[hu] = r < count ? __ldg(p.row_ss + row_base + r) : make_float2(0.f, 0.f);
              }
            }
#pragma unroll
            for (int hu = 0; hu < 4; ++hu)
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                float4& x = v[2 * hu + c];
                x.x = fmaf(x.x, ss[hu].x, ss[hu].y); x.y = fmaf(x.y, ss[hu].x, ss[hu].y);
                x.z = fmaf(x.z, ss[hu].x, ss[hu].y); x.w = fmaf(x.w, ss[hu].x, ss[hu].y);
              }
          }
        }
        const uint32_t it = it_base + (uint32_t)j;
        const uint32_t stage = it % (uint32_t)kXStages;
        const uint32_t phase = (it / (uint32_t)kXStages) & 1u;
        mbar_wait_backoff(&ctl->a_empty[stage], phase ^ 1u, 5 * p.wait_ns);
        tc_fence_after();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          // TMEM column 8(2c+b) + 2t + e of the K block holds feature 16c + 4t + 2b + e (the clip planes in
          // shared memory use the same permutation).  lo = x - hi is exact; the MMA drops its low 13 bits.
          uint32_t rh[16], rl[16];
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const float4 x = v[2 * (2 * h + u) + c];
              split_tf32(x.x, rh[4 * (2 * c) + 2 * u + 0], rl[4 * (2 * c) + 2 * u + 0]);
              split_tf32(x.y, rh[4 * (2 * c) + 2 * u + 1], rl[4 * (2 * c) + 2 * u + 1]);
              split_tf32(x.z, rh[4 * (2 * c + 1) + 2 * u + 0], rl[4 * (2 * c + 1) + 2 * u + 0]);
              split_tf32(x.w, rh[4 * (2 * c + 1) + 2 * u + 1], rl[4 * (2 * c + 1) + 2 * u + 1]);
            }
          const uint32_t ta = a_lane + ((uint32_t)(16 * h) << 16) + stage * 64u;
          tmem_st_16x256b_x4(ta, rh);
          tmem_st_16x256b_x4(ta + 32u, rl);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&ctl->a_full[stage]);
      };
      // this warp's items: j = 2m + par.  Prologue: the first kXRing - 1 of them (one commit group per item,
      // empty groups keep the count uniform)
      const int nmine = (nitems - par + kStageSets - 1) / kStageSets;
#pragma unroll
      for (int m = 0; m < kXRing - 1; ++m) {
        if (m < nmine) issue(m);
        cp_async_commit();
      }
      for (int m = 0; m < nmine; ++m) {
        if (m + kXRing - 1 < nmine) issue((m + kXRing - 1) % kXRing);   // the slot item m - 1 was read from
        cp_async_commit();
        cp_async_wait<kXRing - 1>();                            // item m has landed
        __syncwarp();
        store(kStageSets * m + par, m % kXRing);
        __syncwarp();                                           // every lane is done with the slot
      }
      cp_async_wait<0>();
      it_base += (uint32_t)nitems;
    }
  } else if (warp == kXLoadWarp) {
    // ===================== B loader =====================
    if (lane == 0) {
      uint32_t vi = 0, itb = 0;
      for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
        int e0, count;
        if (kMode == 2) {
          // the 4 videos' pre-packed clip planes (4 KB per video, plane and K block) land side by side: rows 32 v ..
          // 32 v + 31 of the N = 128 operand; a missing video (tail group) re-reads the last one, its columns are ignored
          int g_, row0_;
          item_range(p, n, g_, row0_, count);
          if (count <= 0) continue;
          const uint8_t* base = reinterpret_cast<const uint8_t*>(p.planes);
          for (int t0 = 0; t0 < count; t0 += kXRows) {
            for (int kb = 0; kb < num_kb; ++kb, ++itb) {
              const uint32_t bs = itb % (uint32_t)kXBStages;
              mbar_wait_backoff(&ctl->b_empty[bs], ((itb / (uint32_t)kXBStages) & 1u) ^ 1u, 5 * p.wait_ns);
              mbar_expect_tx(&ctl->b_full[bs], b_buf_bytes);
              for (int v = 0; v < kXGroup; ++v) {
                const int vid = min(g_ * kXGroup + v, p.Nv_real - 1);
                const uint8_t* src = base + ((size_t)vid * num_kb + kb) * 2 * kXBPlane;
                bulk_load(sB + (size_t)bs * b_buf_bytes + (size_t)v * kXBPlane, src, kXBPlane, &ctl->b_full[bs]);
                bulk_load(sB + (size_t)bs * b_buf_bytes + (size_t)(kXGroup + v) * kXBPlane, src + kXBPlane, kXBPlane,
                          &ctl->b_full[bs]);
              }
            }
          }
          continue;
        }
        int vid = n;
        if (kMode == 4) { int r0_; item_range_linear(p, n, vid, r0_, count); }
        else video_range(p, n, e0, count);
        if (count <= 0) continue;
        if (kResB) {
          const uint32_t bb = vi % b_bufs;
          mbar_wait_backoff(&ctl->b_empty[bb], ((vi / b_bufs) & 1u) ^ 1u, 5 * p.wait_ns);
          ++vi;
          mbar_expect_tx(&ctl->b_full[bb], b_buf_bytes);
          const uint8_t* src = reinterpret_cast<const uint8_t*>(p.planes) + (size_t)n * b_buf_bytes;
          for (int kb = 0; kb < num_kb; ++kb)                     // 8 KB per K block: hi plane, lo plane
            bulk_load(sB + (size_t)bb * b_buf_bytes + (size_t)kb * 2 * kXBPlane, src + (size_t)kb * 2 * kXBPlane,
                      2 * kXBPlane, &ctl->b_full[bb]);
        } else {
          // every tile of the video streams the video's row planes again (L2 resident): one stage per K block
          const uint8_t* src = reinterpret_cast<const uint8_t*>(p.planes) + (size_t)vid * num_kb * b_buf_bytes;
          for (int t0 = 0; t0 < count; t0 += kXRows) {
            for (int kb = 0; kb < num_kb; ++kb, ++itb) {
              const uint32_t bs = itb % (uint32_t)kXBStages;
              mbar_wait_backoff(&ctl->b_empty[bs], ((itb / (uint32_t)kXBStages) & 1u) ^ 1u, 5 * p.wait_ns);
              mbar_expect_tx(&ctl->b_full[bs], b_buf_bytes);
              bulk_load(sB + (size_t)bs * b_buf_bytes, src + (size_t)kb * b_buf_bytes, b_buf_bytes, &ctl->b_full[bs]);
            }
          }
        }
      }
    }
  } else if (warp == kXMmaWarp) {
    // ===================== MMA issuer =====================
    const int nb = kMode == 0 ? 32 : p.Npad;                    // UMMA N
    const uint32_t idesc = make_idesc_tf32(nb, kXRows);
    const uint32_t b_plane = (uint32_t)nb * 128u;               // bytes of one plane of one K block
    const bool elected = elect_one();
    const uint64_t bdesc0 = make_smem_desc(smem_u32(sB));
    uint32_t it = 0, vi = 0, tc = 0, itb = 0;
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int e0, count;
      if (kMode == 2) { int g_, r_; item_range(p, n, g_, r_, count); e0 = 0; }
      else if (kMode == 4) { int g_, r_; item_range_linear(p, n, g_, r_, count); e0 = 0; }
      else video_range(p, n, e0, count);
      if (count <= 0) continue;
      uint32_t bb = 0;
      if (kResB) {
        bb = vi % b_bufs;
        mbar_wait_backoff(&ctl->b_full[bb], (vi / b_bufs) & 1u, p.wait_ns);
        ++vi;
      }
      for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
        const uint32_t buf = tc & 1u;
        mbar_wait_backoff(&ctl->tmem_empty[buf], ((tc >> 1) & 1u) ^ 1u, p.wait_ns);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * (uint32_t)kDW;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t stage = it % (uint32_t)kXStages;
          const uint32_t phase = (it / (uint32_t)kXStages) & 1u;
          uint32_t bs = 0;
          if (!kResB) {
            bs = itb % (uint32_t)kXBStages;
            mbar_wait_backoff(&ctl->b_full[bs], (itb / (uint32_t)kXBStages) & 1u, p.wait_ns);
            ++itb;
          }
          mbar_wait_backoff(&ctl->a_full[stage], phase, p.wait_ns);
          tc_fence_after();
          if (elected) {
            const uint32_t a_hi = tmem_base + kXACol0 + stage * 64u;
            const uint32_t a_lo = a_hi + 32u;
            const uint64_t b_hi = kResB ? bdesc0 + (uint64_t)((bb * b_buf_bytes + (uint32_t)kb * 2u * b_plane) >> 4)
                                             : bdesc0 + (uint64_t)((bs * b_buf_bytes) >> 4);
            const uint64_t b_lo = b_hi + (uint64_t)(b_plane >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k) {   // 8 tf32 per MMA: 8 TMEM columns of A, 32 B (+2 x 16 B) of the B swizzle row
              umma_tf32_ts(d_tmem, a_lo + 8 * k, b_hi + 2 * k, idesc, (kb | k) ? 1u : 0u);   // small terms first
              umma_tf32_ts(d_tmem, a_hi + 8 * k, b_lo + 2 * k, idesc, 1u);
              umma_tf32_ts(d_tmem, a_hi + 8 * k, b_hi + 2 * k, idesc, 1u);
            }
            umma_commit(&ctl->a_empty[stage]);
            if (!kResB) umma_commit(&ctl->b_empty[bs]);
          }
          __syncwarp();
        }
        if (elected) umma_commit(&ctl->tmem_full[buf]);
        __syncwarp();
      }
      if (kResB) {
        if (elected) umma_commit(&ctl->b_empty[bb]);
        __syncwarp();
      }
    }
  } else if constexpr (kMode == 2) {
    // ===================== scan: clip windows of kXGroup videos per tile, two groups alternating tiles ================
    // Same per-row arithmetic as mode 0 (sequential window sums, x scale, strict > in proposal order); the 4 videos'
    // dots sit in accumulator columns 32 v .. 32 v + 31.
    const int T = p.T, P = T * (T + 1) / 2;
    const int quarter = warp & 3;
    const uint32_t part = warp >= 2 * kXScanWarps ? 1u : 0u;        // warps 0-3: even tiles, warps 8-11: odd tiles
    const int stid = threadIdx.x;
    uint32_t tc = 0;
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int group, row0, count;
      item_range(p, n, group, row0, count);
      if (count <= 0) continue;
      asm volatile("bar.sync 1, %0;" ::"n"(2 * kXScanWarps * 32) : "memory");   // previous item's tables are dead
      if (part == 0) {
        for (int v = 0; v < kXGroup; ++v) {
          const int vid = min(group * kXGroup + v, p.Nv_real - 1);
          const float* gsc = p.scale + (int64_t)vid * P;
          const int s_ = stid & 31;
          int base = 0;
          for (int w = 1; w <= T; ++w) {
            if ((w & 3) == (stid >> 5) && s_ + w <= T) s_scale[v][(w - 1) * 32 + s_] = __ldg(gsc + base + s_);
            base += T - w + 1;
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(2 * kXScanWarps * 32) : "memory");
      for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
        const uint32_t buf = tc & 1u;
        if (buf != part) continue;
        mbar_wait(&ctl->tmem_full[buf], (tc >> 1) & 1u);
        tc_fence_after();
        const int r = row0 + t0 + quarter * 32 + lane;
#pragma unroll 1
        for (int v = 0; v < kXGroup; ++v) {
          uint32_t raw[32];
          tmem_ld32_issue(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)kDW + (uint32_t)(32 * v), raw);
          tmem_ld_wait();
          if (v == kXGroup - 1) {                 // the accumulator buffer is free once its last slice is in registers
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ctl->tmem_empty[buf]);
          }
          const float* sc = s_scale[v];
          float d[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) d[i] = __uint_as_float(raw[i]);
          float bv0;
          int bi0;
          window_scan_v1<kT32>(d, sc, T, bv0, bi0);
          const int vid = group * kXGroup + v;
          if (r < p.M && t0 + quarter * 32 + lane < count && vid < p.Nv_real) {
            const int64_t o = (int64_t)r * p.ld_out + vid;
            p.out_max[o] = bv0;
            if (p.out_arg) p.out_arg[o] = bi0;
          }
        }
      }
    }
  } else if constexpr (kMode == 0) {
    // ===================== scan: clip windows =====================
    // Thread = tile row.  Windows are visited w-major, so inside each of the 8 independent running maxima
    // (start class s & 7) proposal indices increase and strict > keeps the first maximum; the final merge
    // compares (value desc, index asc).
    const int T = p.T, P = T * (T + 1) / 2;
    const int quarter = warp;
    const int stid = threadIdx.x;                                   // 0..127 among scan threads
    uint32_t tc = 0, vi = 0;
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int e0, count;
      video_range(p, n, e0, count);
      if (count <= 0) continue;
      if constexpr (kDots) {
        // the lane's d[0..32) (zeros beyond T: the clip planes are zero-padded) as eight 16-byte stores, entry order
        for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
          const uint32_t buf = tc & 1u;
          mbar_wait(&ctl->tmem_full[buf], (tc >> 1) & 1u);
          tc_fence_after();
          uint32_t raw[32];
          tmem_ld32_issue(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)kDW, raw);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&ctl->tmem_empty[buf]);
          const int r = t0 + quarter * 32 + lane;
          if (r < count) {
            uint4* dst = reinterpret_cast<uint4*>(p.out_max + (int64_t)(e0 + r) * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = make_uint4(raw[4 * j], raw[4 * j + 1], raw[4 * j + 2], raw[4 * j + 3]);
          }
        }
        continue;
      }
      float* sc = s_scale[vi & 1u];
      // the buffer was last read two videos ago; the barrier below (one per video) orders those reads before
      // these writes: a warp can be at most one video ahead of the slowest one
      {
        const float* gsc = p.scale + (int64_t)n * P;
        const int s_ = stid & 31;
        int base = 0;                                               // p(w, 0)
        for (int w = 1; w <= T; ++w) {
          if ((w & 3) == (stid >> 5) && s_ + w <= T) sc[(w - 1) * 32 + s_] = __ldg(gsc + base + s_);
          base += T - w + 1;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kXScanWarps * 32) : "memory");
      ++vi;
      for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
        const uint32_t buf = tc & 1u;
        mbar_wait(&ctl->tmem_full[buf], (tc >> 1) & 1u);
        tc_fence_after();
        uint32_t raw[32];
        tmem_ld32_issue(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)kDW, raw);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&ctl->tmem_empty[buf]);
        float d[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) d[i] = __uint_as_float(raw[i]);
        float bv0;
        int bi0;
        const int r = t0 + quarter * 32 + lane;
        if constexpr (kT32 && kXTwoPhaseList) {
          float* dcol = sD + quarter * 32 + lane;
          if (kXKnown != 0 && p.known_key) {
            // candidates whose key clip is already fixed: confirm it against the value-only maximum
            const int qi = r < count ? (p.q_list ? p.q_list[e0 + r] : r) : 0;
            const int key = r < count ? __ldg(p.known_key + (int64_t)qi * p.known_ld + n) : 0;
            window_scan_known<kXKnown == 2>(d, sc, dcol, kXRows, key, bv0, bi0);
          } else if (kXListScan != 0) {
            window_scan_v2<kXListScan == 2>(d, sc, dcol, kXRows, bv0, bi0);
          } else {
            window_scan_v1<kT32>(d, sc, T, bv0, bi0);
          }
        } else {
          window_scan_v1<kT32>(d, sc, T, bv0, bi0);
        }
        if (r < count) {
          const int64_t o = p.out_slot ? (int64_t)p.out_slot[e0 + r]
                            : (p.list_stride > 0 ? (int64_t)p.q_list[e0 + r] * p.ld_out + n
                                                 : (p.vid_ptr ? (int64_t)(e0 + r) : (int64_t)r * p.ld_out + n));
          p.out_max[o] = bv0;
          if (p.out_arg) p.out_arg[o] = bi0;
        }
      }
    }
  } else if constexpr (kMode == 4) {
    // ===================== epilogue of the linear layer: + bias, optional ReLU, fp32 store =====================
    // Thread = tile row: its 128 outputs arrive as four 32-column TMEM loads and leave as 16-byte stores.
    const int quarter = warp;
    uint32_t tc = 0;
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int wtile, row0, count;
      item_range_linear(p, n, wtile, row0, count);
      if (count <= 0) continue;
      for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
        const uint32_t buf = tc & 1u;
        mbar_wait(&ctl->tmem_full[buf], (tc >> 1) & 1u);
        tc_fence_after();
        const int r = t0 + quarter * 32 + lane;
        const bool live = r < count;
        float* orow = p.out_max + (int64_t)(row0 + (live ? r : 0)) * p.ld_out;
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t raw[32];
          tmem_ld32_issue(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)kDW + (uint32_t)c0, raw);
          tmem_ld_wait();
          if (c0 == 96) {                          // the accumulator buffer is free once its last slice is in registers
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ctl->tmem_empty[buf]);
          }
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const int col = wtile * 128 + c0 + j;
            if (live && col < p.n_cols) {
              float4 o = make_float4(__uint_as_float(raw[j]), __uint_as_float(raw[j + 1]), __uint_as_float(raw[j + 2]),
                                     __uint_as_float(raw[j + 3]));
              if (p.bias) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col));
                o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
              }
              if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              *reinterpret_cast<float4*>(orow + col) = o;
            }
          }
        }
      }
    }
  } else {
    // ===================== scan: masked max over the rows =====================
    // Thread = tile row: its R dots arrive as 32-column TMEM loads; masked rows score exactly -1e10
    // (mask_logits, method/model.py:444-445); strict > in row order keeps the first maximum (torch.max).
    const int quarter = warp;
    uint32_t tc = 0;
    for (int n = blockIdx.x; n < p.Nv; n += gridDim.x) {
      int e0, count;
      video_range(p, n, e0, count);
      if (count <= 0) continue;
      const uint8_t* mrow = p.mask ? p.mask + (int64_t)n * p.R : nullptr;
      for (int t0 = 0; t0 < count; t0 += kXRows, ++tc) {
        const uint32_t buf = tc & 1u;
        mbar_wait(&ctl->tmem_full[buf], (tc >> 1) & 1u);
        tc_fence_after();
        float bv = -INFINITY;
        int bi = 0;
        for (int c0 = 0; c0 < p.R; c0 += 32) {
          uint32_t raw[32];
          tmem_ld32_issue(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (uint32_t)kDW + (uint32_t)c0, raw);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int r = c0 + j;
            if (r < p.R) {
              float v = __uint_as_float(raw[j]);
              if (mrow && __ldg(mrow + r) == 0) v = DKD_MASKED_SCORE;
              if (v > bv) { bv = v; bi = r; }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&ctl->tmem_empty[buf]);
        const int r = t0 + quarter * 32 + lane;
        if (r < count) {
          const int64_t o = p.out_slot ? (int64_t)p.out_slot[e0 + r]
                                       : (p.vid_ptr ? (int64_t)(e0 + r) : (int64_t)r * p.ld_out + n);
          p.out_max[o] = bv;
          if (p.out_arg) p.out_arg[o] = bi;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kXMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kXTmemCols));
  }
}

// Pre-pack the rows of every video (clips, or frames) into the shared-memory image of the exact kernels' B operand:
// planes[n][kb][plane][rpad rows x 128 B, SWIZZLE_128B], plane 0 = tf32 hi, 1 = tf32 lo, rows >= R zero, features
// of a K block permuted like the A operand (feature 16c + 4t + 2b + e at position 16c + 8b + 2t + e).
__global__ void pack_rows_tf32_kernel(const float* __restrict__ x, int R, int rpad, int D, float* __restrict__ planes,
                                      int64_t total_rows) {
  const int n = blockIdx.x;
  const int num_kb = D / kXKB;
  const uint32_t plane_bytes = (uint32_t)rpad * 128u;
  uint8_t* dst = reinterpret_cast<uint8_t*>(planes) + (size_t)n * num_kb * 2 * plane_bytes;
  for (int i = threadIdx.x; i < num_kb * rpad * 8; i += blockDim.x) {
    const int kb = i / (rpad * 8), rem = i - kb * rpad * 8;
    const int r = rem >> 3, c8 = rem & 7;                           // float4 c8: features 4 c8 .. 4 c8 + 3
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < R && (int64_t)n * R + r < total_rows) v = *reinterpret_cast<const float4*>(x + ((int64_t)n * R + r) * D + kb * kXKB + c8 * 4);
    uint2 h0, l0, h1, l1;
    split_tf32(v.x, h0.x, l0.x); split_tf32(v.y, h0.y, l0.y); split_tf32(v.z, h1.x, l1.x); split_tf32(v.w, h1.y, l1.y);
    const int cc = c8 >> 2, tt = c8 & 3;
    const int p0 = 16 * cc + 2 * tt;                                // b = 0; b = 1 is 8 positions further
    uint8_t* row0 = dst + (size_t)(kb * 2) * plane_bytes;
    uint8_t* d0 = row0 + sw128_off(r, p0 >> 2) + (p0 & 3) * 4;
    uint8_t* d1 = row0 + sw128_off(r, (p0 + 8) >> 2) + (p0 & 3) * 4;
    *reinterpret_cast<uint2*>(d0) = h0;
    *reinterpret_cast<uint2*>(d1) = h1;
    *reinterpret_cast<uint2*>(d0 + plane_bytes) = l0;
    *reinterpret_cast<uint2*>(d1 + plane_bytes) = l1;
  }
}

}  // namespace dkd

using namespace dkd;

static int row_pad(int R, int clip_mode) { return clip_mode ? 32 : ((R + 15) / 16) * 16; }

extern "C" int64_t dkd_clip_planes_bytes(int32_t Nv, int32_t D) {
  if (Nv < 0 || D <= 0 || D % kXKB != 0) return -1;
  return (int64_t)Nv * (D / kXKB) * 2 * kXBPlane;
}
extern "C" int64_t dkd_row_planes_bytes(int32_t Nv, int32_t R, int32_t D) {
  if (Nv < 0 || R <= 0 || R > 128 || D <= 0 || D % kXKB != 0) return -1;
  return (int64_t)Nv * (D / kXKB) * 2 * row_pad(R, 0) * 128;
}

static int pack_rows(const float* x, int32_t Nv, int32_t R, int32_t rpad, int32_t D, float* planes, void* stream) {
  if (!x || !planes || Nv < 0) return DKD_ERR_ARG;
  if (R <= 0 || R > rpad || D <= 0 || D % kXKB != 0 || D > 512) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(planes)) & 15) return DKD_ERR_ALIGN;
  if (Nv == 0) return DKD_OK;
  pack_rows_tf32_kernel<<<Nv, 256, 0, (cudaStream_t)stream>>>(x, R, rpad, D, planes, (int64_t)Nv * R);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}
extern "C" int dkd_pack_clips_tf32(const float* clips, int32_t Nv, int32_t T, int32_t D, float* planes, void* stream) {
  if (T > 32) return DKD_ERR_SHAPE;
  return pack_rows(clips, Nv, T, 32, D, planes, stream);
}
extern "C" int dkd_pack_rows_tf32(const float* xn, int32_t Nv, int32_t R, int32_t D, float* planes, void* stream) {
  if (R > 128) return DKD_ERR_SHAPE;
  return pack_rows(xn, Nv, R, row_pad(R, 0), D, planes, stream);
}

// shared launcher: mode 0 (clip windows; dots: the per-clip dots only) / mode 1 (rows max) / mode 2 / mode 4
static int launch_exact(int mode, ExactParams p, int32_t D, int32_t T, cudaStream_t st, bool dots = false) {
  p.wait_ns = 0u;   // spin: sleeping between polls measured no gain (DESIGN.md section 4)
  int dev = 0, sms = 0, max_smem = 0;
  DKD_CUDA_TRY(cudaGetDevice(&dev));
  DKD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DKD_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const int num_kb = D / kXKB;
  const bool stream0 = mode == 0 && kXStreamB0;                 // mode 0 with the clip planes streamed per K block
  const int ring = stream0 ? DKD_X_RING0 : ((mode == 0 || mode == 2) && D > 448 ? 2 : 3);   // resident B grows with D
  const int ring_warps = mode == 2 ? 4 : kXStageWarps;        // mode 2: one stager warp per TMEM lane quarter
  const int scan_groups = (mode == 0 && kXTwoPhaseList) ? 1 : 0;
  const size_t fixed = sizeof(ExactCtl) + 1024 + 128 + 16384 /* static shared, largest mode */ +
                       (size_t)ring_warps * ring * kXSlotBytes + (size_t)scan_groups * kXScanScratch;
  size_t b_total;
  if (mode == 0 && !stream0) {
    const size_t b_buf = (size_t)num_kb * 2 * kXBPlane;
    if ((size_t)max_smem < fixed + b_buf) return DKD_ERR_SHAPE;
    p.b_bufs = ((size_t)max_smem >= fixed + 2 * b_buf) ? 2 : 1;
    b_total = (size_t)p.b_bufs * b_buf;
  } else {
    p.b_bufs = kXBStages;
    b_total = (size_t)kXBStages * 2 * p.Npad * 128;
    if ((size_t)max_smem < fixed + b_total) return DKD_ERR_SHAPE;
  }
  const size_t smem = fixed - 16384 + b_total;
  const int grid = p.Nv < sms ? p.Nv : sms;
  auto launch = [&](auto kern) -> int {
    DKD_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kXThreads, smem, st>>>(p);
    return DKD_OK;
  };
  int rc;
  if (mode == 0 && dots) {
    if (stream0) rc = launch(exact_umma_kernel<0, true, DKD_X_RING0, true>);
    else rc = (ring == 3) ? launch(exact_umma_kernel<0, true, 3, true>) : launch(exact_umma_kernel<0, true, 2, true>);
  } else if (mode == 0 && stream0) {
    rc = (T == 32) ? launch(exact_umma_kernel<0, true, DKD_X_RING0>) : launch(exact_umma_kernel<0, false, DKD_X_RING0>);
  } else if (mode == 0) {
    if (ring == 3) rc = (T == 32) ? launch(exact_umma_kernel<0, true, 3>) : launch(exact_umma_kernel<0, false, 3>);
    else rc = (T == 32) ? launch(exact_umma_kernel<0, true, 2>) : launch(exact_umma_kernel<0, false, 2>);
  } else if (mode == 2) {
    if (ring == 3) rc = (T == 32) ? launch(exact_umma_kernel<2, true, 3>) : launch(exact_umma_kernel<2, false, 3>);
    else rc = (T == 32) ? launch(exact_umma_kernel<2, true, 2>) : launch(exact_umma_kernel<2, false, 2>);
  } else if (mode == 4) {
    rc = launch(exact_umma_kernel<4, true, 3>);
  } else {
    rc = launch(exact_umma_kernel<1, true, 3>);
  }
  if (rc) return rc;
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_score_max_exact(const float* qn, int32_t M, const float* row_planes, int32_t Nv, int32_t R,
                                   int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg,
                                   int64_t ld_out, const int32_t* vid_ptr, const int32_t* q_list, void* stream) {
  if (!qn || !row_planes || !out_max || M < 0 || Nv < 0) return DKD_ERR_ARG;
  if ((vid_ptr == nullptr) != (q_list == nullptr)) return DKD_ERR_ARG;
  if (R <= 0 || R > 128 || D <= 0 || D % kXKB != 0 || D > 512) return DKD_ERR_SHAPE;
  if (!vid_ptr && ld_out < Nv) return DKD_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(qn) | reinterpret_cast<uintptr_t>(row_planes)) & 15) return DKD_ERR_ALIGN;
  if (M == 0 || Nv == 0) return DKD_OK;
  ExactParams p{};
  p.q = qn; p.M = M; p.planes = row_planes; p.scale = nullptr;
  p.Nv = Nv; p.T = 0; p.D = D; p.R = R; p.Npad = row_pad(R, 0); p.mask = mask;
  p.out_max = out_max; p.out_arg = out_arg; p.ld_out = ld_out;
  p.vid_ptr = vid_ptr; p.vid_cnt = nullptr; p.q_list = q_list; p.out_slot = nullptr;
  return launch_exact(1, p, D, 0, (cudaStream_t)stream);
}

extern "C" int dkd_clip_score_f32(const float* qn, int32_t M, const float* clip_planes, const float* prop_scale,
                                  int32_t Nv, int32_t T, int32_t D, float* out_max, int32_t* out_arg,
                                  int64_t ld_out, const int32_t* vid_ptr, const int32_t* vid_cnt,
                                  const int32_t* q_list, const int32_t* out_slot, const int32_t* known_key,
                                  int64_t known_ld, void* stream) {
  if (!qn || !clip_planes || !prop_scale || !out_max || M < 0 || Nv < 0) return DKD_ERR_ARG;
  if ((vid_ptr == nullptr) != (q_list == nullptr)) return DKD_ERR_ARG;
  if ((out_slot || vid_cnt) && !vid_ptr) return DKD_ERR_ARG;
  if (known_key && (!vid_ptr || known_ld < Nv || T != 32)) return DKD_ERR_ARG;
  if (T <= 0 || T > 32 || D <= 0 || D % kXKB != 0 || D > 512) return DKD_ERR_SHAPE;
  if (!vid_ptr && ld_out < Nv) return DKD_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(qn) | reinterpret_cast<uintptr_t>(clip_planes) | reinterpret_cast<uintptr_t>(prop_scale)) & 15)
    return DKD_ERR_ALIGN;
  if (M == 0 || Nv == 0) return DKD_OK;
  ExactParams p{};
  p.q = qn; p.M = M; p.planes = clip_planes; p.scale = prop_scale;
  p.Nv = Nv; p.T = T; p.D = D; p.R = T; p.Npad = 32; p.mask = nullptr;
  p.out_max = out_max; p.out_arg = out_arg; p.ld_out = ld_out;
  p.vid_ptr = vid_ptr; p.vid_cnt = vid_cnt; p.q_list = q_list; p.out_slot = out_slot;
  p.known_key = known_key; p.known_ld = known_ld;
  if (!vid_ptr && Nv >= kXGroup) {
    // dense form (mode 2): work items = groups of 4 videos x chunks of query tiles, several items per SM
    const int groups = (Nv + kXGroup - 1) / kXGroup;
    const int tiles = (M + kXRows - 1) / kXRows;
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int chunks = 1;
    while (chunks < tiles && (int64_t)groups * chunks < (int64_t)sms * 12) ++chunks;
    p.tiles_per_chunk = (tiles + chunks - 1) / chunks;
    p.tile_chunks = (tiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
    p.Nv_real = Nv;
    p.Nv = groups * p.tile_chunks;
    p.Npad = 128;
    return launch_exact(2, p, D, T, (cudaStream_t)stream);
  }
  return launch_exact(0, p, D, T, (cudaStream_t)stream);
}

// The per-clip dots of the listed pairs (mode-0 list form, dots flag): out_dots[e * 32 + i] = qn[q_list[e]] . clips[n, i]
// for the entries e of video n's CSR run, bit for bit the d[i] dkd_clip_score_f32 scans.  Moment localisation
// (dkd_moment_nms) scans them for every window instead of the maximum alone.
extern "C" int dkd_clip_dots_list(const float* qn, int32_t M, const float* clip_planes, int32_t Nv, int32_t T, int32_t D,
                                  const int32_t* vid_ptr, const int32_t* q_list, float* out_dots, void* stream) {
  if (!qn || !clip_planes || !vid_ptr || !q_list || !out_dots || M < 0 || Nv < 0) return DKD_ERR_ARG;
  if (T <= 0 || T > 32 || D <= 0 || D % kXKB != 0 || D > 512) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(qn) | reinterpret_cast<uintptr_t>(clip_planes) | reinterpret_cast<uintptr_t>(out_dots)) & 15)
    return DKD_ERR_ALIGN;
  if (M == 0 || Nv == 0) return DKD_OK;
  ExactParams p{};
  p.q = qn; p.M = M; p.planes = clip_planes; p.scale = nullptr;
  p.Nv = Nv; p.T = T; p.D = D; p.R = T; p.Npad = 32; p.mask = nullptr;
  p.out_max = out_dots; p.out_arg = nullptr; p.ld_out = 0;
  p.vid_ptr = vid_ptr; p.vid_cnt = nullptr; p.q_list = q_list; p.out_slot = nullptr;
  return launch_exact(0, p, D, T, (cudaStream_t)stream, true);
}

// ---- linear layers of the corpus-side encoder (SURVEY section 8 f1) on the same fp32-grade tensor-core pipeline ----
extern "C" int64_t dkd_weight_planes_bytes(int32_t N, int32_t K) {
  if (N <= 0 || K <= 0 || K % kXKB != 0) return -1;
  return (int64_t)((N + 127) / 128) * (K / kXKB) * 2 * 128 * 128;
}

extern "C" int dkd_pack_weight_tf32(const float* w, int32_t N, int32_t K, float* planes, void* stream) {
  if (!w || !planes || N <= 0) return DKD_ERR_ARG;
  if (K <= 0 || K % kXKB != 0) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(planes)) & 15) return DKD_ERR_ALIGN;
  pack_rows_tf32_kernel<<<(N + 127) / 128, 256, 0, (cudaStream_t)stream>>>(w, 128, 128, K, planes, (int64_t)N);
  DKD_LAUNCH_CHECK();
  return DKD_OK;
}

extern "C" int dkd_linear_exact(const float* x, int64_t M, int32_t K, const float* w_planes, int32_t N,
                                const float* bias, int32_t relu, const float* row_scale_shift, float* out,
                                int64_t ld_out, void* stream) {
  if (!x || !w_planes || !out || M < 0 || N <= 0) return DKD_ERR_ARG;
  if (K <= 0 || K % kXKB != 0 || N % 4 != 0 || ld_out < N || ld_out % 4 != 0 || M > 0x7fffff00LL) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w_planes) | reinterpret_cast<uintptr_t>(out) |
       reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(row_scale_shift)) & 15)
    return DKD_ERR_ALIGN;
  if (M == 0) return DKD_OK;
  ExactParams p{};
  p.q = x; p.M = (int)M; p.planes = w_planes; p.scale = nullptr;
  p.T = 0; p.D = K; p.R = 128; p.Npad = 128; p.mask = nullptr;
  p.out_max = out; p.out_arg = nullptr; p.ld_out = ld_out;
  p.row_ss = reinterpret_cast<const float2*>(row_scale_shift); p.bias = bias; p.relu = relu; p.n_cols = N;
  const int wtiles = (N + 127) / 128;
  const int tiles = (int)((M + kXRows - 1) / kXRows);
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int chunks = 1;
  while (chunks < tiles && (int64_t)wtiles * chunks < (int64_t)sms * 6) ++chunks;
  p.tiles_per_chunk = (tiles + chunks - 1) / chunks;
  p.tile_chunks = (tiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
  p.Nv_real = wtiles;
  p.Nv = wtiles * p.tile_chunks;
  return launch_exact(4, p, K, 0, (cudaStream_t)stream);
}

// Exact clip scores of per-video query lists stored with a fixed stride (the lists dkd_score_max_bf16_lists writes):
// video n owns q_list[n * list_stride, n * list_stride + vid_cnt[n]); entry (q, n) is written into the dense matrices
// at out_max[q * ld_out + n] / out_arg[q * ld_out + n].  Same arithmetic as dkd_clip_score_f32.
extern "C" int dkd_clip_score_list(const float* qn, int32_t M, const float* clip_planes, const float* prop_scale,
                                   int32_t Nv, int32_t T, int32_t D, float* out_max, int32_t* out_arg, int64_t ld_out,
                                   const int32_t* vid_cnt, const int32_t* q_list, int64_t list_stride, void* stream) {
  if (!qn || !clip_planes || !prop_scale || !out_max || !vid_cnt || !q_list || M < 0 || Nv < 0) return DKD_ERR_ARG;
  if (list_stride <= 0 || ld_out < Nv || (int64_t)Nv * list_stride > 0x7fffffffLL) return DKD_ERR_ARG;
  if (T <= 0 || T > 32 || D <= 0 || D % kXKB != 0 || D > 512) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(qn) | reinterpret_cast<uintptr_t>(clip_planes) | reinterpret_cast<uintptr_t>(prop_scale)) & 15)
    return DKD_ERR_ALIGN;
  if (M == 0 || Nv == 0) return DKD_OK;
  ExactParams p{};
  p.q = qn; p.M = M; p.planes = clip_planes; p.scale = prop_scale;
  p.Nv = Nv; p.T = T; p.D = D; p.R = T; p.Npad = 32; p.mask = nullptr;
  p.out_max = out_max; p.out_arg = out_arg; p.ld_out = ld_out;
  p.vid_ptr = nullptr; p.vid_cnt = vid_cnt; p.q_list = q_list; p.out_slot = nullptr; p.list_stride = list_stride;
  return launch_exact(0, p, D, T, (cudaStream_t)stream);
}
