// K2: query x corpus score kernel for sm_100a.
//
//   S[q, v] = sum_k A[q, k] * B[v, k]        A = query operand, B = corpus operand (bf16, K-major)
//
// Persistent, warp-specialised, one CTA per SM:
//   warp 0      TMA producer   (cp.async.bulk.tensor, 128B swizzle, multi-stage smem ring)
//   warp 1      MMA issuer     (tcgen05.mma, fp32 accumulators in TMEM; the warp walks the loop in uniform control
//                              flow, elect.sync picks the issuing lane)
//   warp 2      TMEM allocator (512 columns = two 256-column accumulator slots)
//   warps 4-11  epilogue       (tcgen05.ld, one query row per thread; two warps share each TMEM lane quarter)
// Two epilogues share the main loop:
//   STORE   out = alpha * S                                   (cal_error / sampling pass), written as whole 128-byte
//           row segments through a swizzled shared-memory tile
//   FILTER  per-row window (lo, hi]: count scores above hi, append (score, index) of scores inside
//           the window to a per-row candidate list -- the score matrix never reaches HBM.
//
// Tile shapes (XMVE_TILE overrides the choice made in launch(): 0 / 1 / 2 with the static unit assignment,
// 5 / 4 / 6 the same with the dynamic unit scheduler):
//   SINGLE (0, 5)  one CTA, tcgen05.mma.cta_group::1 of 128 x 256 x 16, two accumulator slots double-buffered (the
//               epilogue of tile i overlaps the MMAs of tile i+1).
//   PAIR (1, 4)  two CTAs of a cluster drive one tcgen05.mma.cta_group::2 of 256 x 256 x 16: each CTA stages its
//               128 query rows and HALF of the corpus tile (32 KB instead of 48 KB per SM and k-block).  Default
//               (with the dynamic scheduler).
//   WIDE (2, 6)  a CTA pair computes 256 queries x 512 corpus rows: per k-block each CTA stages its 128 query rows
//               ONCE plus its halves of TWO corpus sub-tiles and the leader issues two cta_group::2 MMA chains that
//               share the query operand (48 KB per SM per 1024 tensor clocks -- the fewest operand bytes per flop).
//               Both accumulator slots belong to one tile, so the epilogue is not overlapped (kept for experiments:
//               launch() no longer chooses it).
// Unit assignment: static (worker, worker + n_workers, ...) or DYNAMIC -- a scheduler thread (warp 3 of the leader
// CTA) takes the next unit from a global counter and hands it to the producer, MMA and epilogue roles of both CTAs
// through a two-slot shared-memory mailbox, so the units of one corpus tile are always in flight together.
//
// Work is cut into units of ONE corpus tile x a group of query tiles, walked query-tile-major, inside
// super-blocks of the query operand sized for L2 (see plan_schedule()).
//
// Replaces np.dot(l2norm(captions), l2norm(videos).T) in LINAS-engine/evaluation.py:21,45,79 and
// P @ index.T in MultiFusion/src/validate.py:73,90, and (FILTER) the per-row argsort that follows
// them (LINAS-engine/inference.py:79, MultiFusion/src/validate.py:74,92).
#include <cuda.h>
#include <stdlib.h>

#include <atomic>

#include "common.cuh"
#include "ptx_sm100.cuh"

// Dynamic unit scheduler state (DYN kernels): the next unit to hand out.  Every launch takes the next counter of a
// small ring and zeroes it on its own stream first, so launches that overlap on different streams do not share one
// (up to 64 launches in flight).
constexpr int SCHED_RING = 64;
__device__ unsigned long long xmve_sched_next[SCHED_RING];

namespace xmve {
namespace {

constexpr int BM = 128;              // query rows per CTA tile (TMEM lanes)
constexpr int BN = 256;              // corpus rows per accumulator slot (TMEM columns)
constexpr int BK = 64;               // bf16 elements per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int ACC_SLOTS = 2;
constexpr int EPI_WARP0 = 4;
constexpr int TMEM_COLS = ACC_SLOTS * BN;    // 512
constexpr int A_BYTES = BM * BK * 2;         // 16 KB

enum { MODE_STORE = 0, MODE_FILTER = 1 };

// NB = 256-column corpus sub-tiles per tile (1: slots double-buffer, 2: both slots form one tile)
template <bool PAIR, int NB>
struct Cfg {
  static_assert(NB == 1 || (NB == 2 && PAIR), "the wide tile exists for CTA pairs only");
  static constexpr int CTAS = PAIR ? 2 : 1;
  static constexpr int B_ROWS = BN / CTAS;                     // rows of one sub-tile this CTA stages per k-block
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + NB * B_BYTES;   // 48 KB (wide) / 32 KB (pair) / 48 KB (single)
  static constexpr int STAGES = PAIR ? (NB == 2 ? 4 : 6) : 4;
  static constexpr int THREADS = 128 + 256;                    // 4 control warps + 8 epilogue warps
  static constexpr int EPI_COLS = NB == 2 ? BN : BN / 2;       // columns of a slot drained by one epilogue warp:
                                                               // wide: 4 warps per sub-tile; else two warps per
                                                               // TMEM lane quarter split the slot's 256 columns
  static constexpr int PARK_BYTES = (THREADS - 128) * 2 * 8 * 8;   // two lists of STG (score, index) pairs per
                                                                   // epilogue thread (see flush_parked)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + PARK_BYTES;
  static constexpr int LABEL_BYTES = 8 * EPI_COLS;             // labelled FILTER: one label byte per column of the
                                                               // tile, staged per epilogue warp behind the park lists
  static constexpr int SMEM_BYTES_LABELED = SMEM_BYTES + LABEL_BYTES;
  static constexpr int TILE_M = BM * CTAS;                     // query rows per tile
  static constexpr int TILE_N = BN * NB;                       // corpus rows per tile
};

struct Params {
  int64_t nq, nv;
  int k_blocks;
  int m_tiles, n_tiles, m_group, n_mgroups, sb_tiles;   // m_tiles in units of TILE_M rows, n_tiles of TILE_N
  int64_t n_units, units_per_sb;
  uint64_t hint_a, hint_b;
  unsigned long long* sched_next;   // DYN: this launch's unit counter
  // STORE
  float alpha;
  float* out;
  int64_t out_ld;
  int vec_ok;
  // FILTER
  const float* lo;
  const float* hi;
  int32_t* count_above;
  int32_t* cand_count;
  float* cand_score;
  int32_t* cand_idx;
  int32_t cap;
  int defer_append;                 // FILTER: finish a tile's append one tile later (default; XMVE_DEFER=0 disables)
  int single_hit;                   // FILTER: branch-free extraction of a chunk's only candidate (XMVE_SINGLE_HIT=0 disables)
  // labelled FILTER: column v has label labels[v * lab_step] < 64; row q lists only columns whose label bit is set
  // in allow[q] (and counts only those above hi)
  const uint8_t* labels;
  const uint64_t* allow;
  int64_t lab_step;
};

struct Unit {
  int t, mt0, len, rot;   // corpus tile, first query tile, number of query tiles, per-worker rotation
  // i-th query tile of the unit: workers start at different query tiles so that they do not all pull the
  // same query-operand lines out of the same L2 slices at the same time
  __device__ __forceinline__ int mt(int i) const {
    const int j = i + rot;
    return mt0 + (j >= len ? j - len : j);
  }
};
// Units are ordered super-block-major: all (corpus tile, query group) units of the first `sb_tiles` query
// tiles, then the next super-block...  Within a super-block consecutive units share a corpus tile.
// (32-bit arithmetic: launch_cfg() refuses plans of 2^31 units or more; the 64-bit divisions cost the MMA-issuing
// warp a few hundred clocks per unit)
__device__ __forceinline__ Unit decode_unit(const Params& p, int64_t u, int worker) {
  Unit x;
  const uint32_t u32 = static_cast<uint32_t>(u), per_sb = static_cast<uint32_t>(p.units_per_sb);
  const int sb = static_cast<int>(u32 / per_sb);
  const uint32_t r = u32 - static_cast<uint32_t>(sb) * per_sb;
  x.t = static_cast<int>(r / static_cast<uint32_t>(p.n_mgroups));
  const int g = static_cast<int>(r - static_cast<uint32_t>(x.t) * static_cast<uint32_t>(p.n_mgroups));
  const int sb_end = min(p.m_tiles, (sb + 1) * p.sb_tiles);
  x.mt0 = sb * p.sb_tiles + g * p.m_group;
  x.len = max(0, min(sb_end, x.mt0 + p.m_group) - x.mt0);
  x.rot = x.len > 0 ? worker % x.len : 0;
  return x;
}

__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// Candidates found while a TMEM slot is drained are parked in a small per-thread shared-memory list and
// appended to the row's global list AFTER the slot has been handed back to the MMA warp: one atomicAdd per
// thread and tile, issued by all lanes of the warp together, instead of one blocking atomic per candidate
// inside the divergent scan (which cost 25 % of the kernel at ~1e-3 candidates per score; profiles/).
//
// The append is finished ONE TILE LATE: the atomicAdd that reserves the slots is issued right after the tile's
// scan, but its result is first needed when the parked pairs are stored -- after the NEXT tile's scan (the
// lists are double-buffered).  With the stores directly behind the atomic every epilogue warp sat out one L2
// atomic round trip (~1.5 us) per tile, because almost every warp has some lane with a candidate: 3.5-4 us of
// epilogue against 4.4 us of MMA per tile at K = 640 (profiles/r2_summary.md section 6).
constexpr int STG = 8;                                   // parked candidates per thread and list
__device__ __forceinline__ void store_parked(float* cand_score, int32_t* cand_idx, int cap, int64_t row, int base,
                                             const uint2* stg, int n) {
  for (int e = 0; e < n; ++e) {
    const int slot = base + e;
    if (slot < cap) {
      const uint2 c = stg[e];
      cand_score[row * cap + slot] = __uint_as_float(c.x);
      cand_idx[row * cap + slot] = static_cast<int32_t>(c.y);
    }
  }
}
// the blocking form: a list that fills up in the middle of a scan (dense rows; rare)
__device__ __noinline__ void flush_parked(int32_t* cand_count, float* cand_score, int32_t* cand_idx, int cap,
                                          int64_t row, const uint2* stg, int n) {
  const int base = atomicAdd(&cand_count[row], n);
  store_parked(cand_score, cand_idx, cap, row, base, stg, n);
}

struct RowState {
  int64_t row;
  float lo, hi;
  int above;         // scores above hi (count_above)
  int n;             // parked candidates
  uint2* stg;
  uint64_t allow;    // labelled FILTER: label mask of the row
  const uint8_t* lab;   // ... and the labels of the tile's columns this warp drains (shared memory)
};

// labelled FILTER: whether column `i` of the chunk starting at tile column `c` may enter the row's list
__device__ __forceinline__ bool eligible(const RowState& st, int c, int i) {
  return ((st.allow >> st.lab[c + i]) & 1ull) != 0;
}

__device__ __forceinline__ void filter_one(const Params& p, RowState& st, float s, int32_t col) {
  if (s > st.hi) {
    ++st.above;
  } else {
    if (st.n == STG) {
      flush_parked(p.cand_count, p.cand_score, p.cand_idx, p.cap, st.row, st.stg, st.n);
      st.n = 0;
    }
    st.stg[st.n++] = make_uint2(__float_as_uint(s), static_cast<uint32_t>(col));
  }
}

// 32 consecutive scores of one query row: a tree of 3-input maxima decides whether anything enters the
// window (rare); only the 3-element groups whose maximum does are examined element by element.  LABELED: a score
// that entered the window is dropped (neither listed nor counted) unless its column's label is allowed for the row;
// the label is read from shared memory only there, so the cost grows with the hits, not with the scores.
// `c` is the chunk's first column within the warp's share of the tile.
template <bool LABELED>
__device__ __forceinline__ void filter_chunk(const Params& p, const uint32_t (&v)[32], RowState& st, int64_t col,
                                             int c) {
  float m[11];
#pragma unroll
  for (int g = 0; g < 10; ++g)
    m[g] = max3(__uint_as_float(v[3 * g]), __uint_as_float(v[3 * g + 1]), __uint_as_float(v[3 * g + 2]));
  m[10] = fmaxf(__uint_as_float(v[30]), __uint_as_float(v[31]));
  const float a = max3(m[0], m[1], m[2]), b = max3(m[3], m[4], m[5]), cc = max3(m[6], m[7], m[8]);
  if (max3(max3(a, b, cc), m[9], m[10]) > st.lo) {
    const int64_t left = p.nv - col;                     // columns of this chunk inside the corpus
    if (p.single_hit && left >= 32) {
      // Only the lanes with a hit are here (the others wait at the reconvergence point), so what this costs is the
      // length of THEIR instruction stream.  Almost always the chunk holds exactly ONE candidate: count the hits and
      // take the position of the last one without a branch (three independent ALU operations per element) instead
      // of walking eleven group tests, each a branch with its own reconvergence barrier.
      int cnt = 0, pos = 0;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const bool h = __uint_as_float(v[i]) > st.lo;
        cnt += h ? 1 : 0;
        pos = h ? i : pos;
      }
      if (cnt == 1) {                                    // the hit is the chunk's maximum
        if (!LABELED || eligible(st, c, pos))
          filter_one(p, st, max3(max3(a, b, cc), m[9], m[10]), static_cast<int32_t>(col) + pos);
        return;
      }
    }
    const int lim = left < 32 ? static_cast<int>(left) : 32;
#pragma unroll
    for (int g = 0; g < 11; ++g) {
      if (m[g] > st.lo) {
#pragma unroll
        for (int e = 0; e < (g < 10 ? 3 : 2); ++e) {
          const int i = 3 * g + e;
          const float s = __uint_as_float(v[i]);
          if (s > st.lo && i < lim && (!LABELED || eligible(st, c, i)))
            filter_one(p, st, s, static_cast<int32_t>(col) + i);
        }
      }
    }
  }
}

// STORE: 32 rows x 32 columns held one row per lane (the TMEM load layout) go through a 4 KB per-warp shared-memory
// tile so that every global store instruction writes whole 128-byte row segments (a quarter-warp per row) instead of
// 32 scattered 16-byte pieces, one per row: with the direct form the LSU, not the MMA, set the pace of the STORE
// kernels at K = 640 (profiles/r2_summary.md section 7).  16-byte slots are XOR-swizzled by the row so that both the
// row-wise writes and the transposed reads are conflict-free.  All 32 lanes call it; `row0` is lane 0's row.
__device__ __forceinline__ void store_chunk(const Params& p, const uint32_t (&v)[32], int64_t row0, int64_t col,
                                            float4* wbuf, int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    wbuf[lane * 8 + (j ^ (lane & 7))] =
        make_float4(p.alpha * __uint_as_float(v[4 * j]), p.alpha * __uint_as_float(v[4 * j + 1]),
                    p.alpha * __uint_as_float(v[4 * j + 2]), p.alpha * __uint_as_float(v[4 * j + 3]));
  __syncwarp();
  const int jj = lane & 7;
  const int64_t c = col + 4 * jj;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = 4 * i + (lane >> 3);
    const float4 x = wbuf[r * 8 + (jj ^ (r & 7))];
    const int64_t row = row0 + r;
    if (row < p.nq) {
      float* dst = p.out + row * p.out_ld + c;
      if (p.vec_ok && c + 3 < p.nv) {
        *reinterpret_cast<float4*>(dst) = x;
      } else {
        if (c < p.nv) dst[0] = x.x;
        if (c + 1 < p.nv) dst[1] = x.y;
        if (c + 2 < p.nv) dst[2] = x.z;
        if (c + 3 < p.nv) dst[3] = x.w;
      }
    }
  }
  __syncwarp();                                          // the tile is rewritten by the next chunk
}

// COLS columns of one 128-row accumulator slot -> STORE or FILTER (this thread owns query row st.row).  The TMEM
// loads are software-pipelined: chunk c+1 is in flight while chunk c is examined.
// `release()` hands the slot back to the MMA warp.  It is called as soon as the LAST chunk has arrived in registers,
// before that chunk is examined: the accumulator is free from then on, and at K = 640 the MMA warp was waiting for
// this hand-back (profiles/r2b_mma_issue_loop.txt: ~2 try_wait rounds per tile on `tempty`).
template <int MODE, int COLS, bool LABELED, typename Release>
__device__ __forceinline__ void epilogue_slot(const Params& p, uint32_t taddr, RowState& st, int64_t col0,
                                              Release release) {
  const int lane = threadIdx.x & 31;
  uint32_t v0[32], v1[32];
  ptx::tmem_ld_32x32(taddr, v0);
#pragma unroll 1
  for (int c = 0; c < COLS / 32; c += 2) {
    ptx::tmem_ld_wait();
    ptx::tmem_ld_32x32(taddr + (c + 1) * 32, v1);
    if (MODE == MODE_STORE) store_chunk(p, v0, st.row - lane, col0 + c * 32, reinterpret_cast<float4*>(st.stg - lane * 2 * STG), lane);
    else filter_chunk<LABELED>(p, v0, st, col0 + c * 32, c * 32);
    ptx::tmem_ld_wait();
    if (c + 2 < COLS / 32) ptx::tmem_ld_32x32(taddr + (c + 2) * 32, v0);
    else release();
    if (MODE == MODE_STORE) store_chunk(p, v1, st.row - lane, col0 + (c + 1) * 32, reinterpret_cast<float4*>(st.stg - lane * 2 * STG), lane);
    else filter_chunk<LABELED>(p, v1, st, col0 + (c + 1) * 32, (c + 1) * 32);
  }
}

// Unit sequence of one role (producer / MMA issuer / epilogue warp).  Static: worker, worker + n_workers, ...
// Dynamic (DYN): the units are handed out one at a time by a scheduler thread through a two-slot mailbox in shared
// memory, so that the units of one corpus tile are always taken within microseconds of each other -- with the
// static assignment the workers sharing a corpus tile drift apart until each of them re-reads it from DRAM
// (profiles/r1_tile_schedule_sweep.md section 7).
template <bool DYN, bool PAIR>
struct UnitFeed {
  int64_t u, n_units;
  int stride, slot;
  uint32_t phase, rank;
  uint64_t *full, *empty;
  volatile int64_t* box;
  __device__ __forceinline__ void init(int worker, int n_workers, int64_t n_units_, uint64_t* full_, uint64_t* empty_,
                                       int64_t* box_, uint32_t rank_) {
    u = static_cast<int64_t>(worker) - n_workers;
    stride = n_workers;
    n_units = n_units_;
    slot = 0;
    phase = 0;
    full = full_;
    empty = empty_;
    box = box_;
    rank = rank_;
  }
  // Every lane of the calling warp (WARP = true: all 32 lanes call it) or the single calling thread gets the next
  // unit; false at the end.  `arrive`: this thread reports "read" for its role (lane 0 of a warp).
  template <bool WARP>
  __device__ __forceinline__ bool next(bool arrive) {
    if (!DYN) {
      u += stride;
      return u < n_units;
    }
    if (PAIR && rank != 0) ptx::mbar_wait_cluster(&full[slot], phase);
    else ptx::mbar_wait(&full[slot], phase);
    u = box[slot];
    if (WARP) __syncwarp();                                    // ALL lanes have read before lane 0 releases the slot
    if (arrive) {                                              // the slot may be refilled once every role has read it
      // cluster-scope release: the warp's reads of the mailbox must be performed before the leader may refill it
      // (with the default CTA-scope arrive a peer warp busy storing results was seen to read the NEXT unit)
      if (PAIR && rank != 0) ptx::mbar_arrive_remote_release(&empty[slot], 0);
      else ptx::mbar_arrive(&empty[slot]);
    }
    if (++slot == 2) { slot = 0; phase ^= 1; }
    return u < n_units;
  }
};

template <int MODE, bool PAIR, int NB, bool DYN, bool LABELED>
__device__ __forceinline__ void score_body(const CUtensorMap& tm_a, const CUtensorMap& tm_b, const Params& p) {
  using C = Cfg<PAIR, NB>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + ACC_SLOTS;
  uint64_t* sched_full = tempty_bar + ACC_SLOTS;                 // DYN: unit mailbox (2 slots)
  uint64_t* sched_empty = sched_full + 2;
  int64_t* sched_box = reinterpret_cast<int64_t*>(sched_empty + 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sched_box + 2);
  uint2* park = reinterpret_cast<uint2*>(smem + C::STAGES * C::STAGE_BYTES + 256);

  const int warp = threadIdx.x >> 5;   // warp-uniform
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0;      // 0 = leader (issues the pair's MMAs)
  const int n_workers = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int worker = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tm_a);
    ptx::prefetch_tensormap(&tm_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], C::CTAS);                   // one producer arrival per CTA of the pair
      ptx::mbar_init(&empty_bar[s], 1);                        // one tcgen05.commit
    }
    for (int a = 0; a < ACC_SLOTS; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);                        // one tcgen05.commit
      ptx::mbar_init(&tempty_bar[a], (BN / C::EPI_COLS) * 4 * C::CTAS);   // one arrival per warp draining the slot
      ptx::mbar_init(&sched_full[a], 1);                       // the scheduler thread
      ptx::mbar_init(&sched_empty[a], 10 * C::CTAS - (PAIR ? 1 : 0));   // producer + 8 epilogue warps per CTA + MMA
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (PAIR) {
      ptx::tmem_alloc_pair(tmem_slot, TMEM_COLS);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(tmem_slot, TMEM_COLS);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before_sync();
  if (PAIR) ptx::cluster_sync();                               // the peer's barriers exist before anyone signals them
  else __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      UnitFeed<DYN, PAIR> feed;
      feed.init(worker, n_workers, p.n_units, sched_full, sched_empty, sched_box, rank);
      while (feed.template next<false>(true)) {
        const int64_t u = feed.u;
        const Unit un = decode_unit(p, u, worker);
        const int b_row = un.t * C::TILE_N + static_cast<int>(rank) * C::B_ROWS;
        for (int i = 0; i < un.len; ++i) {
          const int a_row = un.mt(i) * C::TILE_M + static_cast<int>(rank) * BM;
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * C::STAGE_BYTES;
            const int kc = kb * BK;
            if (PAIR) {
              // both CTAs' bytes are accounted on the leader's barrier, which expects the pair's total
              if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
              else ptx::mbar_arrive_remote(&full_bar[stage], 0);
              if (p.hint_a) ptx::tma_load_2d_pair_hint(&tm_a, &full_bar[stage], sa, kc, a_row, p.hint_a);
              else ptx::tma_load_2d_pair(&tm_a, &full_bar[stage], sa, kc, a_row);
#pragma unroll
              for (int j = 0; j < NB; ++j) {
                uint8_t* sb = sa + A_BYTES + j * C::B_BYTES;
                if (p.hint_b)
                  ptx::tma_load_2d_pair_hint(&tm_b, &full_bar[stage], sb, kc, b_row + j * BN, p.hint_b);
                else ptx::tma_load_2d_pair(&tm_b, &full_bar[stage], sb, kc, b_row + j * BN);
              }
            } else {
              ptx::mbar_arrive_expect_tx(&full_bar[stage], C::STAGE_BYTES);
              if (p.hint_a) ptx::tma_load_2d_hint(&tm_a, &full_bar[stage], sa, kc, a_row, p.hint_a);
              else ptx::tma_load_2d(&tm_a, &full_bar[stage], sa, kc, a_row);
              if (p.hint_b) ptx::tma_load_2d_hint(&tm_b, &full_bar[stage], sa + A_BYTES, kc, b_row, p.hint_b);
              else ptx::tma_load_2d(&tm_b, &full_bar[stage], sa + A_BYTES, kc, b_row);
            }
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA only) =================
    // The whole warp walks the loop in uniform control flow and one elected lane issues (see umma_bf16_pair_warp).
    if (rank == 0) {
      constexpr uint32_t idesc = ptx::idesc_bf16_f32(C::TILE_M, BN);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      UnitFeed<DYN, PAIR> feed;
      feed.init(worker, n_workers, p.n_units, sched_full, sched_empty, sched_box, rank);
      // low word of the shared-memory descriptors: start address >> 4 | LBO field; stage 0, query operand
      const uint32_t desc0 = static_cast<uint32_t>(ptx::smem_desc_k_sw128(ptx::smem_u32(smem)));
      static_assert(BK / UMMA_K == 4, "umma_bf16_kblock_warp issues four K = 16 MMAs");
      while (feed.template next<true>(lane == 0)) {
        const int64_t u = feed.u;
        const Unit un = decode_unit(p, u, worker);
        for (int i = 0; i < un.len; ++i) {
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            ptx::mbar_wait(&full_bar[stage], phase);           // TMA bytes (of both CTAs) have landed
            ptx::tc_fence_after_sync();
            // (start address field = bytes >> 4; the ring stays inside the field's 256 KB range)
            const uint32_t da = desc0 + static_cast<uint32_t>((stage * C::STAGE_BYTES) >> 4);
#pragma unroll
            for (int j = 0; j < NB; ++j) {
              const int slot = NB == 1 ? acc : j;
              if (kb == 0) {
                ptx::mbar_wait(&tempty_bar[slot], acc_phase ^ 1);   // the epilogue warps have drained this slot
                ptx::tc_fence_after_sync();
              }
              const uint32_t tmem_d = tmem_base + slot * BN;
              const uint32_t db = da + static_cast<uint32_t>((A_BYTES + j * C::B_BYTES) >> 4);
              ptx::umma_bf16_kblock_warp<C::CTAS>(tmem_d, da, db, idesc, kb != 0 ? 1u : 0u);
            }
            // frees the smem slot (in both CTAs) when the MMAs retire
            if (PAIR) ptx::umma_commit_pair_warp(&empty_bar[stage], 0x3);
            else ptx::umma_commit_warp(&empty_bar[stage]);
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
          }
#pragma unroll
          for (int j = 0; j < NB; ++j) {                        // accumulator(s) complete -> epilogue warps
            const int slot = NB == 1 ? acc : j;
            if (PAIR) ptx::umma_commit_pair_warp(&tfull_bar[slot], 0x3);
            else ptx::umma_commit_warp(&tfull_bar[slot]);
          }
          if (NB == 2) acc_phase ^= 1;
          else if (++acc == ACC_SLOTS) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ================================ unit scheduler (DYN, leader CTA) ==============
    if (DYN && lane == 0 && rank == 0) {
      int slot = 0;
      uint32_t phase = 0;
      for (;;) {
        if (PAIR) ptx::mbar_wait_cluster(&sched_empty[slot], phase ^ 1);   // every role of the pair has read this slot
        else ptx::mbar_wait(&sched_empty[slot], phase ^ 1);
        const int64_t u = static_cast<int64_t>(atomicAdd(p.sched_next, 1ull));
        sched_box[slot] = u;
        if (PAIR) {
          ptx::st_remote_u64(&sched_box[slot], 1, static_cast<uint64_t>(u));
          ptx::mbar_arrive_remote_release(&sched_full[slot], 1);
        }
        ptx::mbar_arrive(&sched_full[slot]);
        if (u >= p.n_units) break;                             // the end marker has been handed out too
        if (++slot == 2) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ================================ epilogue ====================================
    const int quarter = warp & 3;                              // TMEM lane quarter this warp may read
    const int grp = (warp - EPI_WARP0) >> 2;                   // wide: sub-tile (slot); else: half of the slot's columns
    const int sub = NB == 2 ? grp : 0;
    const int col_in_slot = NB == 2 ? 0 : grp * C::EPI_COLS;
    const int row_in_tile = static_cast<int>(rank) * BM + quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    RowState st;
    uint2* const lists = park + (threadIdx.x - EPI_WARP0 * 32) * (2 * STG);
    st.stg = lists;
    st.n = 0;
    // labelled FILTER: this warp's label bytes, behind the park lists
    uint8_t* const labs = reinterpret_cast<uint8_t*>(park + (C::THREADS - 128) * 2 * STG) + (warp - EPI_WARP0) * C::EPI_COLS;
    st.lab = labs;
    st.allow = 0;
    // the append of the previous tile that is still to be finished (its atomicAdd is in flight)
    int pend_n = 0, pend_base = 0;
    int64_t pend_row = 0;
    const uint2* pend_stg = lists;
    int acc = 0;
    uint32_t acc_phase = 0;
    UnitFeed<DYN, PAIR> feed;
    feed.init(worker, n_workers, p.n_units, sched_full, sched_empty, sched_box, rank);
    while (feed.template next<true>(lane == 0)) {
      const int64_t u = feed.u;
      const Unit un = decode_unit(p, u, worker);
      const int64_t col0 = static_cast<int64_t>(un.t) * C::TILE_N + sub * BN + col_in_slot;
      for (int i = 0; i < un.len; ++i) {
        const int slot = NB == 1 ? acc : sub;
        st.row = static_cast<int64_t>(un.mt(i)) * C::TILE_M + row_in_tile;
        st.lo = st.hi = __int_as_float(0x7f800000);            // rows past nq: nothing enters the window
        st.above = 0;
        if (MODE == MODE_FILTER && st.row < p.nq) {
          st.lo = p.lo[st.row];
          if (p.hi != nullptr) st.hi = p.hi[st.row];
          if (LABELED) st.allow = p.allow[st.row];
        }
        // labelled FILTER: the loads of the tile's column labels are issued before the wait on the accumulator, so
        // that they complete behind it; the shared-memory copy is read by the hit paths of every lane
        uint32_t lab4 = 0;
        if constexpr (LABELED) {
#pragma unroll
          for (int e = 0; e < C::EPI_COLS / 32; ++e) {
            const int64_t v = col0 + lane * (C::EPI_COLS / 32) + e;
            const uint32_t l = v < p.nv ? p.labels[v * p.lab_step] : 0u;
            lab4 |= l << (8 * e);
          }
        }
        ptx::mbar_wait(&tfull_bar[slot], acc_phase);
        ptx::tc_fence_after_sync();
        if constexpr (LABELED) {
          static_assert(C::EPI_COLS == 128, "labelled FILTER: four label bytes per lane");
          __syncwarp();                                        // every lane is done with the previous tile's labels
          reinterpret_cast<uint32_t*>(labs)[lane] = lab4;
          __syncwarp();
        }
        epilogue_slot<MODE, C::EPI_COLS, LABELED>(p, tmem_base + lane_addr + slot * BN + col_in_slot, st, col0, [&]() {
          ptx::tc_fence_before_sync();
          __syncwarp();                                        // every lane's last TMEM load has completed
          if (lane == 0) {                                     // one arrival per warp on the LEADER's barrier
            if (PAIR && rank != 0) ptx::mbar_arrive_remote(&tempty_bar[slot], 0);
            else ptx::mbar_arrive(&tempty_bar[slot]);
          }
        });
        if (NB == 2) acc_phase ^= 1;
        else if (++acc == ACC_SLOTS) { acc = 0; acc_phase ^= 1; }
        if (MODE == MODE_FILTER) {                             // the slot is already back with the MMA warp
          if (p.defer_append) {
            if (pend_n != 0) store_parked(p.cand_score, p.cand_idx, p.cap, pend_row, pend_base, pend_stg, pend_n);
            pend_n = st.n;
            if (st.n != 0) {
              pend_base = atomicAdd(&p.cand_count[st.row], st.n);   // first read a whole tile from now
              pend_row = st.row;
              pend_stg = st.stg;
              st.stg = st.stg == lists ? lists + STG : lists;
              st.n = 0;
            }
          } else if (st.n != 0) {
            flush_parked(p.cand_count, p.cand_score, p.cand_idx, p.cap, st.row, st.stg, st.n);
            st.n = 0;
          }
          if (st.above != 0 && p.count_above != nullptr) atomicAdd(&p.count_above[st.row], st.above);
        }
      }
    }
    if (MODE == MODE_FILTER && pend_n != 0)
      store_parked(p.cand_score, p.cand_idx, p.cap, pend_row, pend_base, pend_stg, pend_n);
  }

  ptx::tc_fence_before_sync();
  if (PAIR) ptx::cluster_sync();                               // nobody leaves while the peer may still signal it
  else __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after_sync();
    if (PAIR) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int MODE, bool LABELED>
__global__ void __launch_bounds__(Cfg<false, 1>::THREADS, 1)
score_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, false, 1, false, LABELED>(tm_a, tm_b, p);
}

template <int MODE, bool LABELED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<true, 1>::THREADS, 1)
score_pair_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, true, 1, false, LABELED>(tm_a, tm_b, p);
}

template <int MODE, bool LABELED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<true, 2>::THREADS, 1)
score_wide_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, true, 2, false, LABELED>(tm_a, tm_b, p);
}

// the same kernels with the dynamic unit scheduler
template <int MODE, bool LABELED>
__global__ void __launch_bounds__(Cfg<false, 1>::THREADS, 1)
score_dyn_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, false, 1, true, LABELED>(tm_a, tm_b, p);
}

template <int MODE, bool LABELED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<true, 1>::THREADS, 1)
score_pair_dyn_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, true, 1, true, LABELED>(tm_a, tm_b, p);
}

template <int MODE, bool LABELED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<true, 2>::THREADS, 1)
score_wide_dyn_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  score_body<MODE, true, 2, true, LABELED>(tm_a, tm_b, p);
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  static EncodeTiledFn cached = nullptr;
  if (cached == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    XMVE_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (fn == nullptr || qres != cudaDriverEntryPointSuccess)
      return fail(XMVE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cached = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *out = cached;
  return XMVE_OK;
}

// bf16 [rows, k] with row stride `ld` elements -> 2-D tiled map, box = 64 x box_rows, 128B swizzle,
// out-of-bounds elements read as zero.
int make_operand_map(CUtensorMap* map, const void* base, int64_t rows, int64_t k, int64_t ld, int box_rows) {
  EncodeTiledFn encode;
  int s = get_encode_fn(&encode);
  if (s != XMVE_OK) return s;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
  if (const char* env = getenv("XMVE_L2PROMO")) promo = static_cast<CUtensorMapL2promotion>(atoi(env) & 3);
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(XMVE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld k=%lld ld=%lld", static_cast<int>(r),
                static_cast<long long>(rows), static_cast<long long>(k), static_cast<long long>(ld));
  return XMVE_OK;
}

int check_operands(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv, int64_t b_ld,
                   int64_t b_row_step, int k) {
  XMVE_REQUIRE(a_op != nullptr && b_op != nullptr, "score: null operand");
  XMVE_REQUIRE(nq > 0 && nv > 0, "score: empty problem (nq=%lld nv=%lld)", (long long)nq, (long long)nv);
  XMVE_REQUIRE(k > 0 && k % BK == 0, "score: k=%d must be a positive multiple of %d", k, BK);
  XMVE_REQUIRE(a_ld >= k && b_ld >= k && a_ld % 8 == 0 && b_ld % 8 == 0,
               "score: row strides must be >= k and multiples of 8 elements");
  XMVE_REQUIRE(aligned16(a_op) && aligned16(b_op), "score: operands must be 16-byte aligned");
  XMVE_REQUIRE(b_row_step >= 1, "score: b_row_step must be >= 1");
  if (nv > (int64_t(1) << 31) - 2 * BN || nq > (int64_t(1) << 31) - 2 * BM)
    return fail(XMVE_ERR_LIMIT, "score: more than 2^31 rows");
  return XMVE_OK;
}

// L2 plan (round-1 profiles).  About 63 MB of unique data stay in L2 whichever die touches them (a line homed on the
// other die is kept twice), so what must fit is
//   (query operand of the current super-block) + (corpus tiles live across the concurrent workers).
// Queries are walked in super-blocks of <= 40 MB of operand -- 8192 queries x 2048 dims are ONE super-block, so the
// corpus streams from HBM once (measured 9.7 GB for an 8.2 GB operand, +2.8 % over two 16 MB super-blocks) -- and
// inside a super-block several workers share each corpus tile (m_group query tiles each): ~18 MB of corpus tiles live.
void plan_schedule(Params& p, int tile_m, int tile_n, int k, int workers) {
  p.m_tiles = static_cast<int>((p.nq + tile_m - 1) / tile_m);
  p.n_tiles = static_cast<int>((p.nv + tile_n - 1) / tile_n);
  const int64_t a_tile_bytes = static_cast<int64_t>(tile_m) * k * 2;
  int64_t sb_mb = 40;
  if (const char* env = getenv("XMVE_SB_MB")) sb_mb = atoi(env);
  int64_t sbt = (sb_mb << 20) / a_tile_bytes;
  if (sbt < 1) sbt = 1;
  if (sbt > p.m_tiles) sbt = p.m_tiles;
  const int64_t n_sb = (p.m_tiles + sbt - 1) / sbt;
  sbt = (p.m_tiles + n_sb - 1) / n_sb;                       // balance the super-blocks
  int64_t mg = sbt / ((workers + 19) / 20);
  const int64_t balance = (static_cast<int64_t>(p.n_tiles) * sbt) / (static_cast<int64_t>(workers) * 8);
  if (mg > balance) mg = balance;                            // keep >= 8 units per worker for tail balance
  if (const char* env = getenv("XMVE_MGROUP")) mg = atoi(env);
  if (mg < 1) mg = 1;
  if (mg > sbt) mg = sbt;
  p.sb_tiles = static_cast<int>(sbt);
  p.m_group = static_cast<int>(mg);
  p.n_mgroups = static_cast<int>((sbt + mg - 1) / mg);
  p.units_per_sb = static_cast<int64_t>(p.n_tiles) * p.n_mgroups;
  p.n_units = p.units_per_sb * n_sb;
  static const uint64_t hints[4] = {0, ptx::L2_EVICT_LAST, ptx::L2_EVICT_FIRST, ptx::L2_EVICT_NORMAL};
  p.hint_a = p.hint_b = 0;
  if (const char* env = getenv("XMVE_HINT_A")) p.hint_a = hints[atoi(env) & 3];
  if (const char* env = getenv("XMVE_HINT_B")) p.hint_b = hints[atoi(env) & 3];
}

// The next counter of the current device's ring, zeroed on `stream` (shared by every DYN kernel of the process;
// a __device__ symbol has one address per device).
int take_sched_counter(unsigned long long** out, cudaStream_t stream) {
  static void* ring[MAX_DEVICES] = {};
  static std::atomic<unsigned> launch_seq{0};
  const int dev = current_device();
  if (dev < 0) return fail(XMVE_ERR_DEVICE, "score: no current device");
  if (ring[dev] == nullptr) XMVE_CUDA(cudaGetSymbolAddress(&ring[dev], xmve_sched_next));
  *out = static_cast<unsigned long long*>(ring[dev]) + (launch_seq.fetch_add(1) % SCHED_RING);
  XMVE_CUDA(cudaMemsetAsync(*out, 0, sizeof(unsigned long long), stream));
  return XMVE_OK;
}

// (only the selected kernel is instantiated: there is no labelled wide kernel)
template <int MODE, bool LABELED, bool PAIR, int NB, bool DYN>
constexpr auto kernel_for() {
  if constexpr (DYN && !PAIR) return score_dyn_kernel<MODE, LABELED>;
  else if constexpr (DYN && NB == 2) return score_wide_dyn_kernel<MODE, LABELED>;
  else if constexpr (DYN) return score_pair_dyn_kernel<MODE, LABELED>;
  else if constexpr (!PAIR) return score_kernel<MODE, LABELED>;
  else if constexpr (NB == 2) return score_wide_kernel<MODE, LABELED>;
  else return score_pair_kernel<MODE, LABELED>;
}

template <int MODE, bool LABELED, bool PAIR, int NB, bool DYN = false>
int launch_cfg(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv, int64_t b_ld,
               int64_t b_row_step, int k, Params p, cudaStream_t stream) {
  using C = Cfg<PAIR, NB>;
  constexpr int smem_bytes = LABELED ? C::SMEM_BYTES_LABELED : C::SMEM_BYTES;
  static_assert(smem_bytes <= 232448, "more dynamic shared memory than a block may have");
  CUtensorMap tm_a, tm_b;
  int s = make_operand_map(&tm_a, a_op, nq, k, a_ld, BM);
  if (s != XMVE_OK) return s;
  s = make_operand_map(&tm_b, b_op, nv, k, b_ld * b_row_step, C::B_ROWS);
  if (s != XMVE_OK) return s;
  const int sms = sm_count();
  if (sms <= 0) return fail(XMVE_ERR_DEVICE, "score: cannot query the SM count");
  const int workers_max = sms / C::CTAS;
  p.nq = nq;
  p.nv = nv;
  p.k_blocks = k / BK;
  plan_schedule(p, C::TILE_M, C::TILE_N, k, workers_max);
  if (p.n_units >= (int64_t(1) << 31)) return fail(XMVE_ERR_LIMIT, "score: more than 2^31 work units");
  const int workers = static_cast<int>(p.n_units < workers_max ? p.n_units : workers_max);
  const int grid = workers * C::CTAS;
  void (*kern)(const CUtensorMap, const CUtensorMap, const Params) = kernel_for<MODE, LABELED, PAIR, NB, DYN>();
  static bool attr_set[MAX_DEVICES] = {};                     // per <MODE, LABELED, PAIR, NB, DYN> instantiation and device
  const int dev = current_device();
  if (dev < 0) return fail(XMVE_ERR_DEVICE, "score: no current device");
  if (!attr_set[dev]) {
    XMVE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    attr_set[dev] = true;
  }
  if (DYN) {
    int s2 = take_sched_counter(&p.sched_next, stream);
    if (s2 != XMVE_OK) return s2;
  }
  kern<<<grid, C::THREADS, smem_bytes, stream>>>(tm_a, tm_b, p);
  return launch_status(!PAIR ? "score_kernel" : (NB == 2 ? "score_wide_kernel" : "score_pair_kernel"));
}

// Tile choice (measured, profiles/r1_tile_schedule_sweep.md, profiles/r2_summary.md section 7).  The kernel runs at
// the 1 kW power cap, so operand bytes moved per flop decide the sustained rate.  The CTA-pair tile moves a third
// less than the single-CTA tile and, with the DYNAMIC unit scheduler, reads every corpus line from DRAM once (16.4 GB
// for an 8.2 GB operand and two query super-blocks; with the static assignment the workers sharing a corpus tile
// drifted apart and the pair kernels re-read it ~10x): +5 % over the single-CTA tile at realistic candidate
// densities.  The wide tile moves the fewest bytes but cannot overlap its epilogue: since the STORE epilogue writes
// coalesced row segments the pair tile beats it on every STORE shape measured (sampling passes, the 59 800 x 2 990
// evaluation), with the static assignment while both operands stay in L2.
// LABELED (filter only): the wide tile has no shared memory left for the label bytes (2 KB per CTA) and launch()
// never chooses it, so XMVE_TILE=2 / 6 is refused.
template <int MODE, bool LABELED = false>
int launch(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv, int64_t b_ld, int64_t b_row_step,
           int k, Params p, cudaStream_t stream) {
  const int64_t operand_bytes = (nq + nv) * static_cast<int64_t>(k) * 2;
  int tile = (MODE == MODE_STORE && operand_bytes <= (int64_t(48) << 20)) ? 1 : 4;
  if (nq <= BM) tile = 5;   // a handful of queries (AVS, online search): HBM-bound, half of a 256-row query tile is padding
  if (const char* env = getenv("XMVE_TILE")) tile = atoi(env);
  if constexpr (LABELED) {
    if (tile == 2 || tile == 6) return fail(XMVE_ERR_ARG, "score_filter_labeled: the wide tile (XMVE_TILE=%d) has no "
                                            "room for the labels; use 0, 1, 4 or 5", tile);
  } else {
    if (tile == 2) return launch_cfg<MODE, LABELED, true, 2>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
    if (tile == 6)
      return launch_cfg<MODE, LABELED, true, 2, true>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
  }
  if (tile == 1) return launch_cfg<MODE, LABELED, true, 1>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
  if (tile == 4)
    return launch_cfg<MODE, LABELED, true, 1, true>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
  if (tile == 5)
    return launch_cfg<MODE, LABELED, false, 1, true>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
  return launch_cfg<MODE, LABELED, false, 1>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, stream);
}

}  // namespace
}  // namespace xmve

extern "C" int xmve_score_store(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv,
                                int64_t b_ld, int64_t b_row_step, int k, float alpha, float* out, int64_t out_ld,
                                void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  int s = check_operands(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k);
  if (s != XMVE_OK) return s;
  XMVE_REQUIRE(out != nullptr && out_ld >= nv, "score_store: out is null or out_ld < nv");
  Params p{};
  p.alpha = alpha;
  p.out = out;
  p.out_ld = out_ld;
  p.vec_ok = (out_ld % 4 == 0 && aligned16(out)) ? 1 : 0;
  return launch<MODE_STORE>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, static_cast<cudaStream_t>(stream));
}

namespace {
int filter_params(xmve::Params& p, const float* lo, const float* hi, int32_t* count_above, int32_t* cand_count,
                  float* cand_score, int32_t* cand_idx, int32_t cap) {
  XMVE_REQUIRE(lo != nullptr && cand_count != nullptr && cand_score != nullptr && cand_idx != nullptr && cap > 0,
               "score_filter: lo / candidate buffers are required and cap must be > 0");
  XMVE_REQUIRE(hi == nullptr || count_above != nullptr, "score_filter: hi given without count_above");
  p.lo = lo;
  p.hi = hi;
  p.count_above = count_above;
  p.cand_count = cand_count;
  p.cand_score = cand_score;
  p.cand_idx = cand_idx;
  p.cap = cap;
  p.defer_append = 1;
  if (const char* env = getenv("XMVE_DEFER")) p.defer_append = atoi(env) != 0;
  p.single_hit = 1;
  if (const char* env = getenv("XMVE_SINGLE_HIT")) p.single_hit = atoi(env) != 0;
  return XMVE_OK;
}
}  // namespace

extern "C" int xmve_score_filter(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv,
                                 int64_t b_ld, int64_t b_row_step, int k, const float* lo, const float* hi,
                                 int32_t* count_above, int32_t* cand_count, float* cand_score, int32_t* cand_idx,
                                 int32_t cap, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  int s = check_operands(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k);
  if (s != XMVE_OK) return s;
  Params p{};
  s = filter_params(p, lo, hi, count_above, cand_count, cand_score, cand_idx, cap);
  if (s != XMVE_OK) return s;
  return launch<MODE_FILTER>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p, static_cast<cudaStream_t>(stream));
}

extern "C" int xmve_score_filter_labeled(const void* a_op, int64_t nq, int64_t a_ld, const void* b_op, int64_t nv,
                                         int64_t b_ld, int64_t b_row_step, int k, const float* lo, const float* hi,
                                         int32_t* count_above, int32_t* cand_count, float* cand_score,
                                         int32_t* cand_idx, int32_t cap, const uint8_t* labels,
                                         const uint64_t* allow, void* stream) {
  using namespace xmve;
  XMVE_DEVICE_OR_RETURN();
  int s = check_operands(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k);
  if (s != XMVE_OK) return s;
  XMVE_REQUIRE(labels != nullptr && allow != nullptr, "score_filter_labeled: labels and allow are required");
  Params p{};
  s = filter_params(p, lo, hi, count_above, cand_count, cand_score, cand_idx, cap);
  if (s != XMVE_OK) return s;
  p.labels = labels;
  p.allow = allow;
  p.lab_step = b_row_step;
  return launch<MODE_FILTER, true>(a_op, nq, a_ld, b_op, nv, b_ld, b_row_step, k, p,
                                   static_cast<cudaStream_t>(stream));
}
