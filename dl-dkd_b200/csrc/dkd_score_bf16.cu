// bf16 scoring GEMM on tcgen05 tensor cores with a fused max/argmax-over-rows epilogue.
//
//   S[m, (n, r)] = q_bf16[m] . x_bf16[n * R + r]           fp32 accumulate in TMEM
//   out_max[m, n] = max_r S,  out_arg[m, n] = argmax_r   (masked rows = -1e10; among rows equal above the 4 low
//   mantissa bits out_arg is one of them, not always the first: include/dkd_b200.h "Tie rule")
//
// R = L (frame path, method/model.py:318-327) or R = P = 528 clip proposals (SURVEY §8 N3).
//
// Structure (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 8  : TMA producer for the corpus (B) ring — BLOCK_N rows x 64 features per K block
//   warp 9  : tcgen05.mma issuer (one elected lane), accumulators double-buffered in TMEM
//   warp 10 : TMA producer for the query tile (A: 128 queries x D, resident for a whole work
//             item) + TMEM allocation
//   warp 11 : spare
//   warps 0-7: epilogue — two warps per TMEM lane quarter, each owning half of the tile's columns
//             (tcgen05.ld 32x32b.x32/.x16), running top-2 per query row across the R / BLOCK_N tiles
//             of one video; the column position rides in the 4 low mantissa bits of the score
//             (LOP3 + 3 FMNMX per element), the 16-column chunk id is tracked once per chunk.
//             Halves are merged through shared memory; direct fp32 / int32 stores of
//             (max, first argmax, gap to the runner-up) and/or one bit per pair "gap below tau".
// A work item = (query tile of 128, chunk of kVideoChunk videos); items are ordered query-tile
// fastest so that CTAs running at the same time stream the same corpus rows out of L2.
//
// Operand layout: K-major, 128-byte swizzle (TMA SWIZZLE_128B <-> UMMA SWIZZLE_128B descriptors),
// one K block = 64 bf16 = 128 B per row, 8-row groups 1024 B apart.
#include <cstddef>
#include "dkd_umma.cuh"

namespace dkd {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;       // bf16 elements per 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kMaxKBlocks = 8;    // D <= 512
constexpr int kMaxStages = 12;
constexpr int kNumThreads = 384;
// Warp roles.  The issue scheduler favours higher warp ids within an SM sub-partition, so the three
// latency-critical single-lane roles sit above the eight ALU-heavy epilogue warps (0..7).
constexpr int kWarpB = 8, kWarpMma = 9, kWarpA = 10;
constexpr int kTmemCols = 512;

// Running top-2 of "score with its position-in-chunk in the 4 low mantissa bits".
struct Top2 {
  float best, second;
  int chunk;  // 16-column chunk (within the video) that holds `best`
};
constexpr float kNegHuge = -3.0e38f;

// one 16-column chunk: r[0..15] raw fp32 bits, chunk id `cid`.  kTop2 = false (no gap / flag output requested: the frame
// head) tracks the maximum only: LOP3 + FMNMX per element instead of LOP3 + 3 FMNMX — the epilogue, not the tensor
// pipe, bounds the R = 128 problem.
__device__ __forceinline__ bool words_have_zero_byte(const uint4 mw) {
  const uint32_t z = ((mw.x - 0x01010101u) & ~mw.x) | ((mw.y - 0x01010101u) & ~mw.y) |
                     ((mw.z - 0x01010101u) & ~mw.z) | ((mw.w - 0x01010101u) & ~mw.w);
  return (z & 0x80808080u) != 0;
}
// Does the 16-column chunk at mrow (16 mask bytes, 16-byte aligned because R % 16 == 0) hold a masked column?
__device__ __forceinline__ bool chunk_has_masked(const uint8_t* mrow) {
  return words_have_zero_byte(__ldg(reinterpret_cast<const uint4*>(mrow)));
}
// 16-byte read-only load that stays where it is written (volatile asm: issued here, consumed much later)
__device__ __forceinline__ uint4 ldg_nc_v4(const uint8_t* ptr) {
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}

// mrow != nullptr: the chunk has masked columns (their scores become the fill value); nullptr: no masked column —
// the unmasked instruction stream.  The mask depends on (video, column) only, so it is uniform over the warp (lanes
// are query rows) and the branch is divergence free.
template <bool kTop2>
__device__ __forceinline__ void top2_chunk(Top2& t, const uint32_t* r, int cid, const uint8_t* mrow) {
  const float before = t.best;
  if (mrow != nullptr) {
    const uint4 mw = __ldg(reinterpret_cast<const uint4*>(mrow));
    const uint32_t w[4] = {mw.x, mw.y, mw.z, mw.w};
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      uint32_t b = r[j];
      if (((w[j >> 2] >> (8 * (j & 3))) & 0xffu) == 0) b = __float_as_uint(DKD_MASKED_SCORE);
      const float u = __uint_as_float((b & 0xfffffff0u) | (uint32_t)(15 - j));
      if (kTop2) t.second = fmaxf(t.second, fminf(t.best, u));
      t.best = fmaxf(t.best, u);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float u = __uint_as_float((r[j] & 0xfffffff0u) | (uint32_t)(15 - j));
      if (kTop2) t.second = fmaxf(t.second, fminf(t.best, u));
      t.best = fmaxf(t.best, u);
    }
  }
  if (t.best != before) t.chunk = cid;
}

// Instruction descriptor, kind::f16: D=f32, A=B=bf16 (format 1) or IEEE half (format 0), both K-major, M=m, N=n.
__host__ __device__ __forceinline__ uint32_t make_idesc(int n, int m, bool f16) {
  const uint32_t fmt = f16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct GemmParams {
  int M, Mpad, Nv, R, D;
  int block_n;        // columns per MMA tile; R % block_n == 0
  int stages;         // B ring depth
  int kb_per_stage;   // K blocks (64 features) per ring stage / barrier handshake
  int video_chunk;    // videos per work item
  const uint8_t* mask;
  float* out_max;
  int32_t* out_arg;
  float* out_gap;     // optional: best - runner-up (bf16-level ambiguity of the argmax)
  uint32_t* out_flags; // optional: bit (n & 31) of word [m][n >> 5] set when that gap is below `tau`
  float tau;
  int flag_words;     // words per query row = ceil(Nv / 32)
  int32_t* flag_cnt;  // optional: per-video count of pairs whose gap is below tau (caller-zeroed) ...
  int32_t* flag_list; // ... and their query indices, video n at [n * flag_cap, n * flag_cap + flag_cnt[n]) (any order)
  int64_t flag_cap;
  int f16;            // operands are IEEE half instead of bf16 (same 2-byte layout, same MMA kind::f16 rate)
  int64_t ld_out;
  int nv_real;        // kPair kernels: Nv counts video PAIRS and R = 2 x rows per video; nv_real = videos
};

struct __align__(8) SmemCtl {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  // One full / empty pair for the whole resident query tile.  Handing the tile over per K block (slab k of the next
  // item loaded while the last corpus tile still multiplies slabs k+1..) was measured SLOWER (same box, round 2: two-scale
  // GEMM 6.41 -> 6.75 ms, frame head 1.79 -> 1.83 ms): the extra waits / commits sit on the single issuing thread.
  uint64_t a_full, a_empty;
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
  // keep these two LAST: kPair kernels do not allocate them (host: offsetof(SmemCtl, xchg))
  float2 xchg[2][128];  // half-1 -> half-0 epilogue exchange (best, second), double buffered
  int xchg_chunk[2][128];
};

// Final value of one (query m, video v): best / runner-up carry the column position in their 4 low mantissa bits.
__device__ __forceinline__ void emit_result(const GemmParams& p, int m, int v, float b, float s2, int ch) {
  const uint32_t bb = __float_as_uint(b);
  const int idx = (ch << 4) + 15 - (int)(bb & 15u);
  float val = __uint_as_float((bb & 0xfffffff0u) | 8u);
  float sec = __uint_as_float((__float_as_uint(s2) & 0xfffffff0u) | 8u);
  const bool dead = val < -0.99e10f;             // fully masked video: exactly the fill value, first index (torch.max)
  if (dead) val = DKD_MASKED_SCORE;
  const int64_t o64 = (int64_t)m * p.ld_out + v;
  p.out_max[o64] = val;
  if (p.out_arg) p.out_arg[o64] = dead ? 0 : idx;
  const float gap = (s2 <= kNegHuge) ? 3.0e38f : val - sec;
  if (p.out_gap) p.out_gap[o64] = gap;
  if (gap < p.tau) {
    if (p.out_flags) atomicOr(&p.out_flags[(int64_t)m * p.flag_words + (v >> 5)], 1u << (v & 31));
    if (p.flag_list) {
      const int pos = atomicAdd(&p.flag_cnt[v], 1);
      if (pos < p.flag_cap) p.flag_list[(int64_t)v * p.flag_cap + pos] = m;
    }
  }
}

// kCta = 1: one CTA per tile (cta_group::1).  kCta = 2: CTA pair (cluster of 2, cta_group::2): the two CTAs
// hold different query tiles and each half of the corpus tile; the leader (rank 0) issues M=256 MMAs
// that read both halves, which halves the shared-memory operand traffic and the L2->SM corpus traffic
// per CTA and doubles the depth of the corpus ring.
//
// kPair (CTA pairs only; short videos, R <= 128 — the frame head): one MMA tile spans TWO videos (N = 2 R <= 256), CTA
// r of the pair stages video 2 v + r.  The tile's two column halves already belong to the two epilogue warps of every
// TMEM lane quarter, so each warp owns one whole video: no exchange of the halves through shared memory, half the
// accumulator handshakes and half the MMA instructions per video (the R = 128 problem is bound by that per-tile
// overhead, not by the tensor pipe).  The host passes Nv = number of pairs, R = block_n = 2 x rows per video.
template <bool kHasMask, int kCta, bool kTop2, bool kPair>
__global__ void __launch_bounds__(kNumThreads, 1)
score_max_bf16_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                      const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int num_kb = p.D / kBlockK;
  const uint32_t a_kb_bytes = kBlockM * kBlockK * 2;        // 16 KB per K block
  const int b_rows = p.block_n / kCta;                      // corpus rows this CTA stages per K block
  const uint32_t b_kb_bytes = b_rows * kBlockK * 2;         // b_rows x 128 B per K block
  const int kbs = p.kb_per_stage;
  const uint32_t b_stage_bytes = b_kb_bytes * kbs;
  const uint32_t cta_rank = (kCta == 2) ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)num_kb * a_kb_bytes;
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smem_b + (size_t)p.stages * b_stage_bytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_video = p.R / p.block_n;
  const int num_q_tiles = p.Mpad / (kBlockM * kCta);        // query tiles (kCta == 2: tile PAIRS)
  const int num_vchunks = (p.Nv + p.video_chunk - 1) / p.video_chunk;
  const int num_items = num_q_tiles * num_vchunks;
  const int worker = blockIdx.x / kCta;                     // cluster id
  const int num_workers = gridDim.x / kCta;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&ctl->full[i], 1); mbar_init(&ctl->empty[i], 1); }
    mbar_init(&ctl->a_full, 1);
    mbar_init(&ctl->a_empty, 1);
    // tmem_empty: one elected arrive per epilogue warp, from both CTAs of a pair
    for (int i = 0; i < 2; ++i) { mbar_init(&ctl->tmem_full[i], 1); mbar_init(&ctl->tmem_empty[i], 8 * kCta); }
    fence_barrier_init();
  }
  if (warp == kWarpB && lane == 0) { tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_x); }
  if (warp == kWarpA) {
    if (kCta == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctl->tmem_base)), "n"(kTmemCols));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctl->tmem_base)), "n"(kTmemCols));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
  }
  tc_fence_before();
  if (kCta == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = ctl->tmem_base;

  if (warp == kWarpB) {
    // ===== corpus (B) producer =====
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int item = worker; item < num_items; item += num_workers) {
        const int vchunk = item / num_q_tiles;
        const int v0 = vchunk * p.video_chunk;
        const int v1 = min(v0 + p.video_chunk, p.Nv);
        for (int v = v0; v < v1; ++v) {
          for (int t = 0; t < tiles_per_video; ++t) {
            int row = v * p.R + t * p.block_n;
            // odd number of videos: the second half of the last pair stages the last video again (result unused)
            if (kPair && cta_rank == 1 && 2 * v + 1 >= p.nv_real) row -= b_rows;
            for (int kb = 0; kb < num_kb; kb += kbs) {
              mbar_wait(&ctl->empty[stage], phase ^ 1);
              uint8_t* dst = smem_b + (size_t)stage * b_stage_bytes;
              if (kCta == 1) {
                mbar_expect_tx(&ctl->full[stage], b_stage_bytes);
                for (int j = 0; j < kbs; ++j)
                  tma_load_2d(&map_x, &ctl->full[stage], dst + (size_t)j * b_kb_bytes, (kb + j) * kBlockK, row);
              } else {
                // both halves report to the leader's barrier
                if (leader) mbar_expect_tx(&ctl->full[stage], 2 * b_stage_bytes);
                const uint32_t bar = mapa_u32(smem_u32(&ctl->full[stage]), 0);
                for (int j = 0; j < kbs; ++j)
                  tma_load_2d_pair(&map_x, bar, dst + (size_t)j * b_kb_bytes, (kb + j) * kBlockK, row + (int)cta_rank * b_rows);
              }
              if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == kWarpA) {
    // ===== query tile (A) producer =====
    if (lane == 0) {
      uint32_t iphase = 0;
      for (int item = worker; item < num_items; item += num_workers) {
        const int q_tile = (item % num_q_tiles) * kCta + (int)cta_rank;
        mbar_wait(&ctl->a_empty, iphase ^ 1);
        if (kCta == 1) {
          mbar_expect_tx(&ctl->a_full, (uint32_t)num_kb * a_kb_bytes);
          for (int kb = 0; kb < num_kb; ++kb)
            tma_load_2d(&map_q, &ctl->a_full, smem_a + (size_t)kb * a_kb_bytes, kb * kBlockK, q_tile * kBlockM);
        } else {
          if (leader) mbar_expect_tx(&ctl->a_full, 2u * (uint32_t)num_kb * a_kb_bytes);
          const uint32_t bar = mapa_u32(smem_u32(&ctl->a_full), 0);
          for (int kb = 0; kb < num_kb; ++kb)
            tma_load_2d_pair(&map_q, bar, smem_a + (size_t)kb * a_kb_bytes, kb * kBlockK, q_tile * kBlockM);
        }
        iphase ^= 1;
      }
    }
  } else if (warp == kWarpMma) {
    // ===== MMA issuer =====
    if (leader) {
      // The whole warp walks the schedule (converged); one elected lane issues the tcgen05 instructions.
      // The issue path is the critical resource of this kernel (the tensor pipe only queues a few MMAs),
      // so descriptors are built once and advanced with 32-bit immediates, and the wait for the NEXT ring
      // stage is taken while half of the current stage's MMAs are still queued.
      const uint32_t idesc = make_idesc(p.block_n, kBlockM * kCta, p.f16 != 0);
      const bool elected = elect_one();
      const uint64_t adesc0 = make_smem_desc(smem_u32(smem_a));
      const uint64_t bdesc0 = make_smem_desc(smem_u32(smem_b));
      const uint32_t a_kb_step = a_kb_bytes >> 4, b_kb_step = b_kb_bytes >> 4, b_stage_step = b_stage_bytes >> 4;
      int stage = 0; uint32_t phase = 0;
      uint32_t iphase = 0;
      uint32_t tile_ctr = 0;
      const int steps_per_tile = num_kb / kbs;
      long long steps_left = 0;  // ring steps this worker will still consume
      for (int item = worker; item < num_items; item += num_workers) {
        const int v0 = (item / num_q_tiles) * p.video_chunk;
        steps_left += (long long)(min(v0 + p.video_chunk, p.Nv) - v0) * tiles_per_video * steps_per_tile;
      }
      bool have_full = false;  // full[stage] already observed (software-pipelined wait)
      for (int item = worker; item < num_items; item += num_workers) {
        const int vchunk = item / num_q_tiles;
        const int v0 = vchunk * p.video_chunk;
        const int v1 = min(v0 + p.video_chunk, p.Nv);
        mbar_wait(&ctl->a_full, iphase);
        iphase ^= 1;
        tc_fence_after();
        const int ntiles = (v1 - v0) * tiles_per_video;
        for (int tl = 0; tl < ntiles; ++tl, ++tile_ctr) {
          const uint32_t as = tile_ctr & 1u;
          const uint32_t aphase = (tile_ctr >> 1) & 1u;
          mbar_wait(&ctl->tmem_empty[as], aphase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + as * (uint32_t)p.block_n;
          uint64_t adesc = adesc0;
          for (int kb0 = 0; kb0 < num_kb; kb0 += kbs) {
            if (!have_full) mbar_wait(&ctl->full[stage], phase);
            have_full = false;
            tc_fence_after();
            --steps_left;
            int nstage = stage + 1; uint32_t nphase = phase;
            if (nstage == p.stages) { nstage = 0; nphase ^= 1; }
            uint64_t bdesc = bdesc0 + (uint64_t)((uint32_t)stage * b_stage_step);
            for (int j = 0; j < kbs; ++j) {
              if (elected) {
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                  // +2 (16-byte units) = 32 B = 16 bf16 inside the 128 B swizzle row
                  if (kCta == 1) umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb0 | j | k) ? 1u : 0u);
                  else umma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb0 | j | k) ? 1u : 0u);
                }
              }
              adesc += a_kb_step;
              bdesc += b_kb_step;
              // absorb the wait for the NEXT stage behind the MMAs just queued
              if (j == 0 && steps_left > 0) {
                mbar_wait(&ctl->full[nstage], nphase);
                have_full = true;
              }
            }
            if (elected) { if (kCta == 1) umma_commit(&ctl->empty[stage]); else umma_commit_pair(&ctl->empty[stage]); }
            stage = nstage; phase = nphase;
          }
          if (elected) { if (kCta == 1) umma_commit(&ctl->tmem_full[as]); else umma_commit_pair(&ctl->tmem_full[as]); }
        }
        if (elected) { if (kCta == 1) umma_commit(&ctl->a_empty); else umma_commit_pair(&ctl->a_empty); }
      }
    }
  } else if (warp < 8) {
    // ===== epilogue =====
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may read
    const int half = warp >> 2;                   // column half of every tile
    const int row_in_tile = quarter * 32 + lane;
    const int chunks = p.block_n >> 4;
    const int c_lo = half == 0 ? 0 : ((chunks + 1) >> 1);            // first 16-col chunk of this half
    const int c_hi = half == 0 ? ((chunks + 1) >> 1) : chunks;       // one past the last
    uint32_t tile_ctr = 0;
    uint32_t vctr = 0;
    for (int item = worker; item < num_items; item += num_workers) {
      const int q_tile = (item % num_q_tiles) * kCta + (int)cta_rank;
      const int vchunk = item / num_q_tiles;
      const int v0 = vchunk * p.video_chunk;
      const int v1 = min(v0 + p.video_chunk, p.Nv);
      const int m = q_tile * kBlockM + row_in_tile;
      if constexpr (kPair) {
        // one whole video per warp: column half `half` of pair v is video 2 v + half
        const int rr = p.R >> 1;                    // rows per video
        const int nch = rr >> 4;                    // 16-column chunks per video (<= 8)
        uint32_t mbits_next = 0;
        for (int v = v0; v < v1; ++v, ++tile_ctr) {
          const int vr = 2 * v + half;
          Top2 t2;
          t2.best = kNegHuge; t2.second = kNegHuge; t2.chunk = 0;
          const uint8_t* mvid = kHasMask ? p.mask + (int64_t)min(vr, p.nv_real - 1) * rr : nullptr;
          // which of the video's chunks hold masked columns: lane c looks at chunk c, BEFORE the wait for the
          // accumulator, so the load's latency hides behind it (one dependent mask load per chunk inside the tile
          // made the epilogue, not the tensor pipe, pace the R = 128 problem)
          uint32_t mbits = 0;
          uint4 mw_next = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
          if (kHasMask) {
            mbits = v == v0 ? __ballot_sync(0xffffffffu, lane < nch && chunk_has_masked(mvid + (lane << 4))) : mbits_next;
            // the NEXT video's mask bytes are requested now and looked at after this tile: their latency overlaps
            // the tile's TMEM loads instead of sitting in front of the next accumulator wait
            if (v + 1 < v1 && lane < nch)
              mw_next = ldg_nc_v4(p.mask + (int64_t)min(vr + 2, p.nv_real - 1) * rr + (lane << 4));
          }
          const uint32_t as = tile_ctr & 1u;
          const uint32_t aphase = (tile_ctr >> 1) & 1u;
          mbar_wait(&ctl->tmem_full[as], aphase);
          tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * (uint32_t)p.block_n +
                                 (uint32_t)(half * rr);
          // two rounds of <= 4 chunks: 64 accumulator registers in flight instead of 128
#pragma unroll 1
          for (int c0 = 0; c0 < nch; c0 += 4) {
            uint32_t r[64];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int c = c0 + 2 * i;
              if (c + 1 < nch) tmem_ld32_issue(taddr + (uint32_t)(c << 4), r + 32 * i);
              else if (c < nch) tmem_ld16_issue(taddr + (uint32_t)(c << 4), r + 32 * i);
            }
            tmem_ld_wait();
            if (c0 + 4 >= nch) {
              // the last columns of the tile are in registers: hand the accumulator back to the MMA warp BEFORE the
              // max / argmax work on them (with two accumulators the tile period is (MMA + epilogue hold time) / 2)
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&ctl->tmem_empty[as]), 0));
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int c = c0 + i;
              if (c < nch) top2_chunk<kTop2>(t2, r + 16 * i, c, (kHasMask && ((mbits >> c) & 1u)) ? mvid + (c << 4) : nullptr);
            }
          }
          if (vr < p.nv_real && m < p.M) emit_result(p, m, vr, t2.best, t2.second, t2.chunk);
          if (kHasMask) mbits_next = __ballot_sync(0xffffffffu, words_have_zero_byte(mw_next));
        }
      } else {
      for (int v = v0; v < v1; ++v, ++vctr) {
        Top2 t2;
        t2.best = kNegHuge; t2.second = kNegHuge; t2.chunk = 0;
        const uint8_t* mvid = kHasMask ? p.mask + (int64_t)v * p.R : nullptr;
        for (int t = 0; t < tiles_per_video; ++t, ++tile_ctr) {
          const uint32_t as = tile_ctr & 1u;
          const uint32_t aphase = (tile_ctr >> 1) & 1u;
          mbar_wait(&ctl->tmem_full[as], aphase);
          tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * (uint32_t)p.block_n;
          const int cid0 = t * chunks;  // chunk id (within the video) of this tile's first chunk
          // All TMEM loads of this warp's column half are issued back to back and waited for ONCE:
          // tcgen05.ld latency is long while the tensor pipe is busy, so it is paid per tile, not per chunk.
          uint32_t r[96];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const int c = c_lo + 2 * i;
            if (c + 1 < c_hi) tmem_ld32_issue(taddr + (uint32_t)(c << 4), r + 32 * i);
            else if (c < c_hi) tmem_ld16_issue(taddr + (uint32_t)(c << 4), r + 32 * i);
          }
          tmem_ld_wait();
          // The tile's columns are in registers: hand the accumulator back to the MMA warp BEFORE the max / argmax work
          // (with two accumulators the tile period is max(MMA, (MMA + epilogue hold time) / 2)).  Measured: 1-2 % back
          // to back, nothing when the chip is cool — at N = 176 the kernel is bound by the board's power cap, not by
          // this hold time (profiles/r2_ab_gemm_items.md); for the masked R = 128 pair tiles above it was the limiter.
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (kCta == 1) mbar_arrive(&ctl->tmem_empty[as]);
            else mbar_arrive_cluster(mapa_u32(smem_u32(&ctl->tmem_empty[as]), 0));
          }
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const int c = c_lo + i;
            if (c < c_hi) {
              const uint8_t* mrow = kHasMask ? mvid + ((cid0 + c) << 4) : nullptr;
              if (kHasMask && !chunk_has_masked(mrow)) mrow = nullptr;
              top2_chunk<kTop2>(t2, r + 16 * i, cid0 + c, mrow);
            }
          }
        }
        // merge the two column halves of this query row (named barrier per lane quarter, 64 threads)
        const int slot = vctr & 1u;
        if (half == 1) {
          ctl->xchg[slot][row_in_tile] = make_float2(t2.best, t2.second);
          ctl->xchg_chunk[slot][row_in_tile] = t2.chunk;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(quarter + 1) : "memory");
        if (half == 0) {
          const float2 o = ctl->xchg[slot][row_in_tile];
          const int oc = ctl->xchg_chunk[slot][row_in_tile];
          // candidates in column order within equal scores: compare (value desc, chunk asc)
          float b = t2.best, s2 = t2.second;
          int ch = t2.chunk;
          const bool take = (o.x > b) || (o.x == b && oc < ch);
          s2 = fmaxf(fmaxf(s2, o.y), take ? b : o.x);
          if (take) { b = o.x; ch = oc; }
          if (m < p.M) emit_result(p, m, v, b, s2, ch);
        }
      }
      }  // !kPair
    }
  }

  tc_fence_before();
  if (kCta == 2) cluster_sync_all(); else __syncthreads();
  if (warp == kWarpA) {
    tc_fence_after();
    if (kCta == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

// ---- host side ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

static int make_map_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                       bool f16) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return DKD_ERR_DRIVER;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? DKD_OK : DKD_ERR_DRIVER;
}

// Largest multiple of 16 that divides R and is <= 192 (each epilogue warp holds <= 96 columns in registers).
static int pick_block_n(int R) {
  for (int n = 192; n >= 16; n -= 16)
    if (R % n == 0) return n;
  return 0;
}

}  // namespace dkd

using namespace dkd;

template <bool kHasMask, int kCta, bool kTop2, bool kPair = false>
static int launch_gemm(const CUtensorMap& map_q, const CUtensorMap& map_x, const GemmParams& p, int grid,
                       size_t smem_bytes, cudaStream_t st) {
  auto kern = score_max_bf16_kernel<kHasMask, kCta, kTop2, kPair>;
  DKD_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCta;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DKD_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, map_q, map_x, p));
  return DKD_OK;
}

static int score_max_tc(const uint16_t* q_bf16, int32_t M, int32_t Mpad, const uint16_t* x_bf16,
                        int32_t Nv, int32_t R, int32_t D, const uint8_t* mask, float* out_max,
                        int32_t* out_arg, float* out_gap, int64_t ld_out, uint32_t* out_flags,
                        float tau, void* stream, bool f16, int32_t* flag_cnt = nullptr, int32_t* flag_list = nullptr,
                        int64_t flag_cap = 0) {
  if (!q_bf16 || !x_bf16 || !out_max || M < 0 || Nv < 0 || ld_out < Nv) return DKD_ERR_ARG;
  if ((flag_cnt == nullptr) != (flag_list == nullptr) || (flag_list && flag_cap <= 0)) return DKD_ERR_ARG;
  if (Mpad < M || Mpad % kBlockM != 0) return DKD_ERR_SHAPE;
  if (R <= 0 || R > 4096 || R % 16 != 0 || D <= 0 || D % kBlockK != 0 || D / kBlockK > kMaxKBlocks) return DKD_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(q_bf16) & 15) || (reinterpret_cast<uintptr_t>(x_bf16) & 15)) return DKD_ERR_ALIGN;
  if (M == 0 || Nv == 0) return DKD_OK;
  if ((int64_t)Nv * R > 0x7fffffffLL) return DKD_ERR_SHAPE;
  if (mask && (reinterpret_cast<uintptr_t>(mask) & 15)) return DKD_ERR_ALIGN;   // 16-byte mask loads per chunk

  int dev = 0, sms = 0, max_smem = 0;
  DKD_CUDA_TRY(cudaGetDevice(&dev));
  DKD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DKD_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));

  // Short videos (R <= 128: the frame head) on CTA pairs: one N = 2 R tile spans two videos (kPair kernels).
#ifdef DKD_NO_PAIR_TILES     // A/B builds only (tools/build_variant.sh)
  const bool pair = false;
#else
  const bool pair = R <= 128 && Nv >= 2 && Mpad % (2 * kBlockM) == 0 && sms >= 2;
#endif
  const int block_n = pair ? 2 * R : pick_block_n(R);
  if (block_n == 0) return DKD_ERR_SHAPE;

  // CTA pairs (cta_group::2) whenever the shapes allow: two query tiles per pair, corpus tile split in
  // halves of a multiple of 8 rows.
  const int cta = (Mpad % (2 * kBlockM) == 0 && (block_n / 2) % 8 == 0 && sms >= 2) ? 2 : 1;

  const int num_kb = D / kBlockK;
  const size_t a_bytes = (size_t)num_kb * kBlockM * kBlockK * 2;
  // K blocks per ring stage.  Every stage costs one full/empty handshake on the single issuing thread,
  // which is the scarce resource: CTA pairs (half-size stages) take 3 K blocks per stage when D allows,
  // measured 1.38 PF vs 1.05 PF with 1 (profiles/r1_gemm_variants.md).  Pair tiles stage R <= 128 rows per CTA and
  // issue N <= 256 instructions (twice the tensor time per handshake): 2 K blocks per stage keep >= 4 stages.
  int kbs = 1;
  if (cta == 2) kbs = (num_kb % 3 == 0 && !(pair && R > 88)) ? 3 : ((num_kb % 2 == 0) ? 2 : 1);
#ifdef DKD_PAIR_KBS          // A/B builds only
  if (pair && num_kb % DKD_PAIR_KBS == 0) kbs = DKD_PAIR_KBS;
#endif
#ifdef DKD_MAIN_KBS          // A/B builds only (2 K blocks per stage at N = 176: 6.5 -> 7.1 ms, profiles/r2_ab_gemm_items.md)
  if (!pair && cta == 2 && num_kb % DKD_MAIN_KBS == 0) kbs = DKD_MAIN_KBS;
#endif
  const size_t b_stage = (size_t)(block_n / cta) * kBlockK * 2 * kbs;
  // pair tiles never exchange column halves: without the exchange buffers (the tail of SmemCtl) a fourth 32 KB stage fits
  const size_t ctl_bytes = pair ? offsetof(SmemCtl, xchg) : sizeof(SmemCtl);
  const size_t fixed = a_bytes + ctl_bytes + 1024 /* alignment slack */ + 256;
  if ((size_t)max_smem < fixed + 2 * b_stage) return DKD_ERR_SHAPE;
  int stages = (int)(((size_t)max_smem - fixed) / b_stage);
  if (stages > kMaxStages) stages = kMaxStages;
  const size_t smem_bytes = fixed + (size_t)stages * b_stage;

  CUtensorMap map_q, map_x;
  int rc = make_map_2d(&map_q, q_bf16, (uint64_t)Mpad, (uint64_t)D, kBlockM, f16);
  if (rc) return rc;
  rc = make_map_2d(&map_x, x_bf16, (uint64_t)Nv * R, (uint64_t)D, (uint32_t)(block_n / cta), f16);
  if (rc) return rc;

  GemmParams p{};
  p.M = M; p.Mpad = Mpad; p.D = D; p.block_n = block_n; p.stages = stages; p.kb_per_stage = kbs;
  p.nv_real = Nv;
  const int nv_items = pair ? (Nv + 1) / 2 : Nv;     // scheduling unit: a video, or a pair of videos
  p.Nv = nv_items; p.R = pair ? 2 * R : R;
  p.f16 = f16 ? 1 : 0;
  p.mask = mask; p.out_max = out_max; p.out_arg = out_arg; p.out_gap = out_gap; p.ld_out = ld_out;
  p.out_flags = out_flags; p.tau = tau; p.flag_words = (Nv + 31) / 32;
  p.flag_cnt = flag_cnt; p.flag_list = flag_list; p.flag_cap = flag_cap;
  // videos (pairs) per work item: enough items for every worker (CTA or CTA pair) x several waves, >= 1.  Longer
  // items (fewer reloads of the resident query tile) were tried — 24 / 32 / 40 / 51 / 64 videos, also a cost model that
  // avoids a ragged last round: interleaved in one process they are all within 2 % of 16, and 64 is 5 % slower
  // (profiles/r2_ab_gemm_items.md).
  const int num_q_tiles = Mpad / (kBlockM * cta);
  const int workers = sms / cta;
  int vc = 16;
  while (vc > 1 && (int64_t)num_q_tiles * ((nv_items + vc - 1) / vc) < (int64_t)workers * 8) vc >>= 1;
  p.video_chunk = vc;
  const int64_t num_items = (int64_t)num_q_tiles * ((nv_items + vc - 1) / vc);
  const int grid = (int)(num_items < workers ? num_items : workers) * cta;

  cudaStream_t st = (cudaStream_t)stream;
  const bool top2 = out_gap || out_flags || flag_list;      // the runner-up is tracked only when somebody reads it
  if (pair) {   // pair == true implies cta == 2 (R % 16 == 0)
    if (top2) return mask ? launch_gemm<true, 2, true, true>(map_q, map_x, p, grid, smem_bytes, st)
                          : launch_gemm<false, 2, true, true>(map_q, map_x, p, grid, smem_bytes, st);
    return mask ? launch_gemm<true, 2, false, true>(map_q, map_x, p, grid, smem_bytes, st)
                : launch_gemm<false, 2, false, true>(map_q, map_x, p, grid, smem_bytes, st);
  }
  if (top2) {
    if (cta == 2) return mask ? launch_gemm<true, 2, true>(map_q, map_x, p, grid, smem_bytes, st)
                              : launch_gemm<false, 2, true>(map_q, map_x, p, grid, smem_bytes, st);
    return mask ? launch_gemm<true, 1, true>(map_q, map_x, p, grid, smem_bytes, st)
                : launch_gemm<false, 1, true>(map_q, map_x, p, grid, smem_bytes, st);
  }
  if (cta == 2) return mask ? launch_gemm<true, 2, false>(map_q, map_x, p, grid, smem_bytes, st)
                            : launch_gemm<false, 2, false>(map_q, map_x, p, grid, smem_bytes, st);
  return mask ? launch_gemm<true, 1, false>(map_q, map_x, p, grid, smem_bytes, st)
              : launch_gemm<false, 1, false>(map_q, map_x, p, grid, smem_bytes, st);
}

extern "C" int dkd_score_max_bf16(const uint16_t* q_bf16, int32_t M, int32_t Mpad, const uint16_t* x_bf16,
                                  int32_t Nv, int32_t R, int32_t D, const uint8_t* mask, float* out_max,
                                  int32_t* out_arg, float* out_gap, int64_t ld_out, uint32_t* out_flags,
                                  float tau, void* stream) {
  return score_max_tc(q_bf16, M, Mpad, x_bf16, Nv, R, D, mask, out_max, out_arg, out_gap, ld_out, out_flags, tau,
                      stream, false);
}

extern "C" int dkd_score_max_f16(const uint16_t* q_f16, int32_t M, int32_t Mpad, const uint16_t* x_f16,
                                 int32_t Nv, int32_t R, int32_t D, const uint8_t* mask, float* out_max,
                                 int32_t* out_arg, float* out_gap, int64_t ld_out, uint32_t* out_flags,
                                 float tau, void* stream) {
  return score_max_tc(q_f16, M, Mpad, x_f16, Nv, R, D, mask, out_max, out_arg, out_gap, ld_out, out_flags, tau,
                      stream, true);
}

// The GEMM with the ambiguous-pair lists written straight from the epilogue (no bit matrix, no dkd_select_flagged
// pass): flag_cnt (Nv, caller-zeroed) counts the pairs of every video whose best / runner-up gap is below tau,
// flag_list holds their query indices, video n at [n * flag_cap, n * flag_cap + flag_cnt[n]).  flag_cap >= M makes
// overflow impossible.  Feed the lists to dkd_clip_score_list (dense scatter of the exact results).
extern "C" int dkd_score_max_bf16_lists(const uint16_t* q, int32_t M, int32_t Mpad, const uint16_t* x, int32_t Nv,
                                        int32_t R, int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg,
                                        int64_t ld_out, float tau, int32_t* flag_cnt, int32_t* flag_list,
                                        int64_t flag_cap, int32_t f16_operands, void* stream) {
  if (!flag_cnt || !flag_list || !out_arg) return DKD_ERR_ARG;
  return score_max_tc(q, M, Mpad, x, Nv, R, D, mask, out_max, out_arg, nullptr, ld_out, nullptr, tau, stream,
                      f16_operands != 0, flag_cnt, flag_list, flag_cap);
}
