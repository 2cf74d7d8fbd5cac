// pagerank.cu — PageRank over the device in-CSR.
//
// Replaces crates/algos/src/page_rank.rs:58-168 (`page_rank`, `page_rank_iteration`).
//
// Two schedules (gb_pr_mode, include/graph_b200.h):
//   EXACT  — the reference's sweep as one thread executes it: in place, CSR-order f32 sums, separate
//            multiply/add (no FMA), IEEE division.  One warp walks the vertices in id order; lanes
//            only parallelise the gather loads, the additions stay sequential.  Bit-exact with the
//            reference wherever the reference is deterministic (n <= 16384 = one chunk).
//   JACOBI — the throughput path (double-buffered, deterministic).
//
// JACOBI design (round 2).  A pull sweep issues one 4-byte gather per edge, and divergent gathers
// that miss L1 are limited to ~1 per clock per SM by the L1TEX->XBAR request port
// (profiles/r01_gather_ceiling_microbench.txt) — 27 % of the HBM roofline, whatever the layout of the
// index stream.  Shared memory serves ~9 random 4-byte reads per clock.  So the sweep is COLUMN
// BLOCKED: vertices are renumbered by in-degree descending, then out-degree descending (hot sources
// first); the source vector is cut into blocks of B entries that fit in shared memory, and every
// (row, block) pair that is expected to hold at least tau edges gets a SEGMENT of 16-bit block-local
// source ids in that block's stream.  A persistent CTA brings a block into shared memory with TMA bulk
// copies (cp.async.bulk + mbarrier), then its warps stream the segments (coalesced 128-bit loads, 8 ids per lane), gather from
// shared memory, and reduce lanes that belong to the same row with a segmented warp scan; one f32
// partial per (row, block) pair goes back to HBM.  Edges of pairs below the threshold (and all edges
// of short rows) stay in a SELL-32 layout with 32-bit ids: one lane per row, gathers through L1/L2
// (no shared memory: the whole 228 KB serve as L1); that kernel also completes every row whose
// segments lie in at most 4 blocks.  A finish kernel adds the hub rows' partials in a fixed order
// (f64), applies the update of page_rank.rs:148-158 and reduces the sweep error.
// Everything is deterministic: bit-identical run to run for a given shard count; across shard counts the
// ranks agree to ~2e-7 (DESIGN.md §2).
//
// Multi-GPU (1-D edge-cut by destination): the 32-row slices of the internal order are dealt
// round-robin to the P ranks, so every rank holds the same mix of hub and tail rows; a rank builds the
// layout of its own rows only and stores each finished out_score into every peer's next vector
// (multimem.st through the NVSwitch when a multicast mapping is given, else one store per peer).
//
// Algorithmic bytes per sweep: 4m (targets) + 4(n+1) (offsets) + 5*4n (out_scores read+write,
// scores read+write, out-degree read) = 4m + 24n + 4  (BASELINE.md §3).
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <numeric>

#include "common.cuh"

namespace gb {

constexpr int PR_WARPS = 32;        // warps per CTA of the sweep kernels: one persistent CTA per SM
constexpr int PR_THREADS = PR_WARPS * 32;
constexpr int PR_SELL_THREADS = 512; // SELL kernel: two 16-warp CTAs per SM and no shared memory (L1 keeps it all)
constexpr int PR_FIN_THREADS = 256;
constexpr uint32_t PR_MAX_PROFILE_EVENTS = 256;  // sweeps bracketed by CUDA events when profiling is on
constexpr uint32_t CB_G = 4;                 // block-local ids per group (one 64-bit load per lane)
constexpr uint32_t CB_BLOCK_DEFAULT = 49152; // source-vector entries per block (192 KB of shared memory)
constexpr uint32_t CB_BLOCK_MAX = 56 * 1024;
constexpr double CB_TAU_DEFAULT = 1.5;       // a (row, block) pair gets a segment if it expects >= tau edges
constexpr uint32_t CB_MAX_BLOCKS = 8192;     // hot blocks kept (the staircase rarely needs more than ~1000)
constexpr uint32_t CB_TASK_CHUNKS = 32;      // chunks per task (one per warp)
constexpr uint32_t SELL_FEW = 4;             // rows with segments in at most this many blocks are finished by k_pr_sell itself
constexpr uint32_t FIN_CTA_BLOCKS = 64;      // finish: 32-row groups with segments in more blocks get a CTA each
constexpr uint32_t CB_NONE = 0xFFFFFFFFu;
constexpr uint32_t CB_MEGA_DEG = 32768;      // layout build: rows with more in-edges go through one stable radix sort
constexpr uint32_t CB_MEGA_JBITS = 14;       // key = row << 14 | block rank (0x3FFF = not in a segment)
constexpr uint32_t CB_ILP = 4;               // 32-edge batches in flight per warp in the layout build
// chunk flags (bits 24.. of PrChunk.w)
constexpr uint32_t CB_HEAD_CONT = 1u, CB_TAIL_CONT = 2u, CB_INTERIOR = 4u;

// ---- the cyclic deal of 32-row slices over the ranks of the 1-D edge-cut ---------------------------
struct PrDeal {
  uint32_t P = 1, p = 0;
};
__host__ __device__ __forceinline__ uint32_t deal_global(uint32_t l, uint32_t P, uint32_t p) {
  return (((l >> 5) * P + p) << 5) | (l & 31u);
}
// number of local rows whose global index is below R
static inline uint32_t deal_count(uint32_t R, uint32_t P, uint32_t p) {
  const uint32_t F = R >> 5, rem = R & 31u;
  const uint32_t full = F > p ? (F - p + P - 1) / P : 0;
  uint32_t c = full * 32;
  if (rem && (F % P) == p) c += rem;
  return c;
}

struct PrPlan {
  uint32_t n = 0;
  uint32_t n_active = 0;  // global rows with in-degree > 0 (renumbered to [0, n_active))
  uint64_t m = 0;
  PrDeal deal;
  uint32_t n_loc = 0;     // local active rows
  uint32_t n_cb = 0;      // local rows [0, n_cb) own at least one column-block segment
  uint64_t loc_edges = 0; // in-edges of the local rows
  uint64_t cb_edges = 0;  // of which served from column blocks
  DevBuf<uint32_t> new_id;    // old id -> internal id
  DevBuf<uint32_t> outdeg;    // out-degree by internal id [n]
  // column blocks
  uint32_t B = 0, KB = 0;       // block entries, hot blocks
  uint64_t S = 0;               // staircase size = sum of nrows[j]
  uint64_t NG = 0;              // groups in all block streams
  uint32_t chunk_groups = 0, n_chunks = 0, n_tasks = 0, n_fix = 0;
  uint32_t fix_max_row = 0;     // largest local row that owns a segment cut by a chunk boundary
  DevBuf<uint32_t> blk;         // [KB] source block of hot rank j
  DevBuf<uint32_t> nrows;       // [KB] local rows [0, nrows[j]) have a segment in block j (non-increasing)
  DevBuf<uint32_t> poff;        // [KB+1] staircase offsets
  DevBuf<uint2> cb_ids;         // [NG] groups of 4 block-local 16-bit ids (pad id = B)
  DevBuf<uint32_t> cb_bits;     // [NG/32 + 4] bit g set <=> group g starts a segment
  DevBuf<float> partial;        // [S] one partial sum per (block, row) pair
  DevBuf<uint4> chunks;         // [n_chunks] (g_begin, g_end, row_before, j | flags << 24)
  DevBuf<uint32_t> tail_slot;   // [n_chunks] staircase slot of the segment cut by the chunk end
  DevBuf<double> side;          // [2 n_chunks] head / tail parts of segments cut by chunk boundaries
  DevBuf<uint32_t> fix_list;    // [n_fix] chunks whose tail segment continues in later chunks
  DevBuf<uint2> tasks;          // [n_tasks] (first chunk, chunk count | block rank << 8), fattest blocks first
  DevBuf<uint32_t> task_ctr;    // [grid_cb] per-range task cursors (reset by the finish kernel)
  DevBuf<float> rem;            // [n_cb] SELL remainder sums of the rows that also have segments
  DevBuf<uint32_t> fin_kb;      // [ceil(n_cb / 32)] blocks of the first row of each 32-row group (finish kernel)
  // SELL-32 (all local active rows; rows < n_cb hold only the edges outside their segments)
  uint32_t num_slices = 0;
  DevBuf<uint4> sell;         // slice-major, then 4-edge group, then lane
  DevBuf<uint2> slice_meta;   // per slice: (first uint4 index, uint4 groups per lane)
  // state (single-GPU path; the shard API brings its own vectors)
  DevBuf<float> x[2];
  DevBuf<float> scores;
  unsigned grid_cb = 0, grid_sell = 0, grid_fin = 1;
  uint32_t n_fin_warp = 0;   // rows [0, n_fin_warp) own segments in more than FIN_CTA_BLOCKS blocks
  uint32_t fin_u = 4;        // finish: row groups per warp iteration (template argument of k_pr_finish)
  uint32_t fin_hub_ctas = 0; // finish CTAs that take the hub groups (the others take rows [n_fin_warp, n_fin))
  uint32_t n_fin = 0;        // rows [0, n_fin) are completed by k_pr_finish, [n_fin, n_cb) by k_pr_sell
  uint32_t few_nrows[SELL_FEW] = {}, few_poff[SELL_FEW] = {};
  DevBuf<double> block_err;  // per CTA error partials (SELL CTAs, then finish CTAs)
  DevBuf<double> err_hist;   // error of each sweep of the current batch
  DevBuf<uint32_t> ctrl;     // [0] = done flag (sweep number at which tolerance was met), [1] = ticket
  size_t smem_cb = 0;
  std::vector<cudaEvent_t> prof_events;
  // GB_PR_TRACE=1 (diagnostics): CUDA events between the kernels of every sweep; averages are printed
  // to stderr when the layout is released
  bool trace = false;
  mutable std::vector<cudaEvent_t> trace_events;  // 5 per traced sweep
  uint64_t bytes() const {
    return new_id.bytes() + outdeg.bytes() + blk.bytes() + nrows.bytes() + poff.bytes() + cb_ids.bytes() +
           cb_bits.bytes() + partial.bytes() + chunks.bytes() + tail_slot.bytes() + side.bytes() +
           fix_list.bytes() + tasks.bytes() + rem.bytes() + fin_kb.bytes() + sell.bytes() + slice_meta.bytes() + x[0].bytes() +
           x[1].bytes() + scores.bytes() + block_err.bytes() + err_hist.bytes();
  }
};

void free_pr_plan(PrPlan* p) {
  if (!p) return;
  if (p->trace && p->trace_events.size() >= 5) {
    cudaDeviceSynchronize();
    double acc[4] = {0, 0, 0, 0};
    const size_t sweeps = p->trace_events.size() / 5;
    for (size_t i = 0; i < sweeps; ++i)
      for (int k = 0; k < 4; ++k) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p->trace_events[5 * i + k], p->trace_events[5 * i + k + 1]);
        acc[k] += ms;
      }
    fprintf(stderr, "[gb trace] shard %u/%u, %zu sweeps: k_pr_cb %.4f  k_pr_fixup %.4f  k_pr_sell %.4f  k_pr_finish %.4f ms\n",
            p->deal.p, p->deal.P, sweeps, acc[0] / sweeps, acc[1] / sweeps, acc[2] / sweeps, acc[3] / sweeps);
  }
  for (cudaEvent_t e : p->trace_events) cudaEventDestroy(e);
  for (cudaEvent_t e : p->prof_events) cudaEventDestroy(e);
  delete p;
}
uint64_t pr_plan_bytes(const PrPlan* p) { return p ? p->bytes() : 0; }

// ---- small device helpers --------------------------------------------------------------------
__device__ __forceinline__ uint4 ld_stream_u4(const uint32_t* p) {
  uint4 r;  // streamed once per sweep: keep it out of L1 so the gathered vector stays there
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ld_stream_u2(const uint2* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
__device__ __forceinline__ uint32_t warp_max(uint32_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
  return v;
}

// ---- plan construction kernels ---------------------------------------------------------------
__global__ void k_perm_keys(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ out_off,
                            uint32_t n, uint64_t* __restrict__ keys, uint32_t* __restrict__ ids) {
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    uint32_t indeg = in_off[v + 1] - in_off[v];
    uint32_t outdeg = out_off[v + 1] - out_off[v];
    // in-degree descending (hub rows first, rows of similar length become neighbours), then
    // out-degree descending (hot sources first inside equal in-degrees).  R-MAT's expected in- and
    // out-degree of a vertex coincide, so this is also a hot-first order of the SOURCES.
    keys[v] = ((uint64_t)(uint32_t)(~indeg) << 32) | (uint32_t)(~outdeg);
    ids[v] = v;
  }
}
__global__ void k_perm_scatter(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ out_off,
                               const uint32_t* __restrict__ in_off, uint32_t n, uint32_t* __restrict__ new_id,
                               uint32_t* __restrict__ outdeg, uint32_t* __restrict__ indeg) {
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += gridDim.x * blockDim.x) {
    if (r == n) {
      indeg[n] = 0;
      continue;
    }
    uint32_t v = sorted_ids[r];
    new_id[v] = r;
    outdeg[r] = out_off[v + 1] - out_off[v];
    indeg[r] = in_off[v + 1] - in_off[v];
  }
}
__global__ void k_count_active(const uint32_t* __restrict__ indeg, uint32_t n, uint32_t* __restrict__ count) {
  uint32_t act = 0;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) act += indeg[r] > 0;
  for (int o = 16; o > 0; o >>= 1) act += __shfl_xor_sync(0xFFFFFFFFu, act, o);
  if ((threadIdx.x & 31) == 0 && act) atomicAdd(count, act);
}
// out-edges leaving each source block (one CTA per block): the block's share of all gathers
__global__ void k_blk_edges(const uint32_t* __restrict__ outdeg, uint32_t n, uint32_t B,
                            unsigned long long* __restrict__ blk_edges) {
  __shared__ unsigned long long part[8];
  const uint32_t b = blockIdx.x;
  const uint64_t lo = (uint64_t)b * B, hi = min((uint64_t)n, lo + B);
  unsigned long long s = 0;
  for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) s += outdeg[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (uint32_t w = 0; w < blockDim.x / 32; ++w) t += part[w];
    blk_edges[b] = t;
  }
}
// rows_ge[b] = number of (global) rows with in-degree >= dmin[b] (indeg is non-increasing)
__global__ void k_rows_ge(const uint32_t* __restrict__ indeg, uint32_t n_active, const uint32_t* __restrict__ dmin,
                          uint32_t nblk, uint32_t* __restrict__ rows_ge) {
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += gridDim.x * blockDim.x) {
    const uint32_t d = dmin[b];
    uint32_t lo = 0, hi = n_active;  // first index with indeg < d
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (indeg[mid] >= d) lo = mid + 1;
      else hi = mid;
    }
    rows_ge[b] = lo;
  }
}

// Classification of the in-edges of the rows that own segments (local rows [n_mega, n_cb)).  An edge
// from source s (internal id) lands in block s / B; if that block is hot (rank j) and the row is inside
// the block's row prefix it belongs to segment (j, row), else to the row's SELL remainder.  One warp walks
// a row in CSR order and leaves one 8-byte RECORD per edge, so that the fill pass — which has to wait for
// the scan over all segment sizes — is a plain scatter with no lookups left:
//   segment edge:   x = block-local id | j << 16,   y = 1 << 31 | position inside the segment
//   remainder edge: x = internal source id,         y = position inside the row's SELL lane
// Positions follow the CSR order (the per-pair counter is advanced batch by batch, each batch waits for
// the previous one's counter value): the layout is deterministic.
constexpr uint32_t CB_REC_SEG = 0x80000000u;
template <bool CHECK>
__device__ __forceinline__ uint32_t cb_classify_row(uint32_t l, uint32_t b0, uint32_t d, uint32_t n,
                                                    const uint32_t* __restrict__ in_tgt,
                                                    const uint32_t* __restrict__ new_id,
                                                    const uint32_t* __restrict__ hot_of_blk,
                                                    const uint32_t* __restrict__ nrows,
                                                    const uint32_t* __restrict__ poff,
                                                    const uint32_t* __restrict__ blk, uint32_t B,
                                                    uint32_t* __restrict__ cnt, uint2* __restrict__ rec, uint32_t lane) {
  uint32_t rem = 0;
  // CB_ILP batches of 32 edges per iteration: their dependent loads (target -> internal id -> block
  // rank -> row prefix) are issued together, so a long row's single warp is not latency bound
  for (uint32_t i = 0; i < d; i += 32 * CB_ILP) {
    uint32_t j[CB_ILP], src[CB_ILP];
    bool valid[CB_ILP];
#pragma unroll
    for (uint32_t u = 0; u < CB_ILP; ++u) {
      const uint32_t k = i + 32 * u + lane;
      valid[u] = k < d;
      src[u] = 0;
      if (valid[u]) {
        uint32_t t = in_tgt[b0 + k];
        if (CHECK && t >= n) t = 0;  // reported by k_feed_check; keep the lookups in range meanwhile
        src[u] = new_id[t];
      }
    }
#pragma unroll
    for (uint32_t u = 0; u < CB_ILP; ++u) j[u] = valid[u] ? hot_of_blk[src[u] / B] : CB_NONE;
#pragma unroll
    for (uint32_t u = 0; u < CB_ILP; ++u)
      if (j[u] != CB_NONE && l >= nrows[j[u]]) j[u] = CB_NONE;
#pragma unroll
    for (uint32_t u = 0; u < CB_ILP; ++u) {
      const bool cb = j[u] != CB_NONE;
      const uint32_t peers = __match_any_sync(0xFFFFFFFFu, j[u]);
      const uint32_t leader = (uint32_t)__ffs(peers) - 1u;
      uint32_t base = 0, local = 0;
      if (cb) {
        local = src[u] - blk[j[u]] * B;
        if (lane == leader) base = atomicAdd(cnt + poff[j[u]] + l, (uint32_t)__popc(peers));
      }
      base = __shfl_sync(0xFFFFFFFFu, base, leader);  // also orders this batch's counter update before the next
      const uint32_t rb = __ballot_sync(0xFFFFFFFFu, valid[u] && !cb);
      if (cb) {
        rec[b0 + i + 32 * u + lane] = make_uint2(local | (j[u] << 16), CB_REC_SEG | (base + __popc(peers & ((1u << lane) - 1u))));
      } else if (valid[u]) {
        rec[b0 + i + 32 * u + lane] = make_uint2(src[u], rem + __popc(rb & ((1u << lane) - 1u)));
      }
      rem += __popc(rb);
    }
  }
  return rem;
}
// rows in internal order (the whole in-CSR is resident): one warp per local row
__global__ void k_cb_count(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ in_tgt,
                           const uint32_t* __restrict__ old_of, const uint32_t* __restrict__ new_id,
                           const uint32_t* __restrict__ hot_of_blk, const uint32_t* __restrict__ nrows,
                           const uint32_t* __restrict__ poff, const uint32_t* __restrict__ blk, uint32_t B,
                           uint32_t row0, uint32_t n_cb, PrDeal deal, uint32_t* __restrict__ cnt,
                           uint2* __restrict__ rec, uint32_t* __restrict__ lens,
                           unsigned long long* __restrict__ cb_edges) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long in_cb = 0;
  for (uint32_t l = row0 + warp; l < n_cb; l += nwarps) {
    const uint32_t old = old_of[deal_global(l, deal.P, deal.p)];
    const uint32_t b0 = in_off[old], d = in_off[old + 1] - b0;
    const uint32_t rem = cb_classify_row<false>(l, b0, d, 0u, in_tgt, new_id, hot_of_blk, nrows, poff, blk, B, cnt, rec, lane);
    if (lane == 0) {
      lens[l] = rem;
      in_cb += d - rem;
    }
  }
  if (lane == 0 && in_cb) atomicAdd(cb_edges, in_cb);
}
// rows [v0, v1) in ORIGINAL order (a chunk of the in-CSR that has just arrived over PCIe): a warp takes
// 32 consecutive rows, keeps those that are local and own segments, and walks them one after the other
__global__ void k_cb_count_rows(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ in_tgt,
                                const uint32_t* __restrict__ new_id, const uint32_t* __restrict__ hot_of_blk,
                                const uint32_t* __restrict__ nrows, const uint32_t* __restrict__ poff,
                                const uint32_t* __restrict__ blk, uint32_t B, uint32_t v0, uint32_t v1, uint32_t n,
                                uint32_t row0, uint32_t n_cb, PrDeal deal, uint32_t* __restrict__ cnt,
                                uint2* __restrict__ rec, uint32_t* __restrict__ lens,
                                unsigned long long* __restrict__ cb_edges) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long in_cb = 0;
  for (uint64_t base = (uint64_t)v0 + 32ull * warp; base < v1; base += 32ull * nwarps) {
    const uint64_t v = base + lane;
    uint32_t l = CB_NONE, b0 = 0, d = 0;
    if (v < v1) {
      const uint32_t gid = new_id[v], slice = gid >> 5;
      if (slice % deal.P == deal.p) {
        const uint32_t loc = ((slice / deal.P) << 5) | (gid & 31u);
        if (loc >= row0 && loc < n_cb) {
          l = loc;
          b0 = in_off[v];
          d = in_off[v + 1] - b0;
        }
      }
    }
    uint32_t todo = __ballot_sync(0xFFFFFFFFu, l != CB_NONE);
    while (todo) {
      const int src_lane = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t rl = __shfl_sync(0xFFFFFFFFu, l, src_lane);
      const uint32_t rb = __shfl_sync(0xFFFFFFFFu, b0, src_lane);
      const uint32_t rd = __shfl_sync(0xFFFFFFFFu, d, src_lane);
      const uint32_t rem = cb_classify_row<true>(rl, rb, rd, n, in_tgt, new_id, hot_of_blk, nrows, poff, blk, B, cnt, rec, lane);
      if (lane == 0) {
        lens[rl] = rem;
        in_cb += rd - rem;
      }
    }
  }
  if (lane == 0 && in_cb) atomicAdd(cb_edges, in_cb);
}
// range check of a chunk of targets and of the offsets of its rows (what validate_device_targets does
// for a resident CSR)
__global__ void k_feed_check(const uint32_t* __restrict__ tgt, uint64_t count, uint32_t n, unsigned int* __restrict__ bad) {
  unsigned int mine = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
    mine += tgt[i] >= n;
  if (mine) atomicAdd(bad, mine);
}
__global__ void k_feed_monotone(const uint32_t* __restrict__ off, uint32_t n, unsigned int* __restrict__ bad) {
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
    if (off[v] > off[v + 1]) atomicAdd(bad, 1u);
}
// ---- the longest rows (a prefix of the local rows) go through ONE stable radix sort -----------------
// A row's warp walks it 128 edges at a time, ~3 us per step: a million-edge hub would take tens of
// milliseconds on its own.  Its edges are instead keyed (row << 14 | block rank), sorted stably — so
// the edges of one (row, block) pair end up contiguous AND in CSR order — and counted / placed from the
// sorted sequence, one thread per edge.
__global__ void k_mega_deg(const uint32_t* __restrict__ indeg, uint32_t n_mega, PrDeal deal, uint32_t* __restrict__ out) {
  for (uint32_t l = blockIdx.x * blockDim.x + threadIdx.x; l < n_mega; l += gridDim.x * blockDim.x)
    out[l] = indeg[deal_global(l, deal.P, deal.p)];
}
__global__ void k_mega_keys(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ in_tgt,
                            const uint32_t* __restrict__ old_of, const uint32_t* __restrict__ new_id,
                            const uint32_t* __restrict__ hot_of_blk, const uint32_t* __restrict__ nrows, uint32_t B,
                            const uint32_t* __restrict__ moff, uint32_t n_mega, uint32_t M, PrDeal deal,
                            uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = n_mega;  // row with moff[row] <= i < moff[row + 1]
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) / 2;
      if (moff[mid] <= i) lo = mid;
      else hi = mid;
    }
    const uint32_t l = lo;
    const uint32_t old = old_of[deal_global(l, deal.P, deal.p)];
    const uint32_t src = new_id[in_tgt[in_off[old] + (i - moff[l])]];
    uint32_t j = hot_of_blk[src / B];
    if (j != CB_NONE && l >= nrows[j]) j = CB_NONE;
    keys[i] = (l << CB_MEGA_JBITS) | (j == CB_NONE ? (1u << CB_MEGA_JBITS) - 1u : j);
    vals[i] = src;
  }
}
__global__ void k_mega_starts(const uint32_t* __restrict__ keys, uint32_t M, uint32_t* __restrict__ start) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x)
    start[i] = (i == 0 || keys[i] != keys[i - 1]) ? i : 0u;  // max-scanned into "first index of my run"
}
__global__ void k_mega_counts(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ start, uint32_t M,
                              const uint32_t* __restrict__ poff, uint32_t* __restrict__ cnt,
                              uint32_t* __restrict__ lens, unsigned long long* __restrict__ cb_edges) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
    if (i + 1 < M && keys[i + 1] == keys[i]) continue;  // not the last edge of its run
    const uint32_t len = i + 1 - start[i];
    const uint32_t l = keys[i] >> CB_MEGA_JBITS, j = keys[i] & ((1u << CB_MEGA_JBITS) - 1u);
    if (j == (1u << CB_MEGA_JBITS) - 1u) {
      lens[l] = len;
    } else {
      cnt[poff[j] + l] = len;
      atomicAdd(cb_edges, (unsigned long long)len);
    }
  }
}
__global__ void k_mega_fill(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                            const uint32_t* __restrict__ start, uint32_t M, const uint32_t* __restrict__ poff,
                            const uint32_t* __restrict__ blk, uint32_t B, const uint32_t* __restrict__ goff,
                            uint16_t* __restrict__ ids, const uint2* __restrict__ slice_meta,
                            uint32_t* __restrict__ sell) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
    const uint32_t pos = i - start[i];
    const uint32_t l = keys[i] >> CB_MEGA_JBITS, j = keys[i] & ((1u << CB_MEGA_JBITS) - 1u);
    if (j == (1u << CB_MEGA_JBITS) - 1u) {
      const uint2 meta = slice_meta[l >> 5];
      sell[((uint64_t)meta.x + (uint64_t)(pos / 4) * 32 + (l & 31u)) * 4 + (pos % 4)] = vals[i];
    } else {
      ids[(uint64_t)goff[poff[j] + l] * CB_G + pos] = (uint16_t)(vals[i] - blk[j] * B);
    }
  }
}
__global__ void k_lens_tail(const uint32_t* __restrict__ indeg, uint32_t n_cb, uint32_t n_loc, PrDeal deal,
                            uint32_t* __restrict__ lens) {
  for (uint32_t l = n_cb + blockIdx.x * blockDim.x + threadIdx.x; l < n_loc; l += gridDim.x * blockDim.x)
    lens[l] = indeg[deal_global(l, deal.P, deal.p)];
}
__global__ void k_loc_edges(const uint32_t* __restrict__ indeg, uint32_t n_loc, PrDeal deal,
                            unsigned long long* __restrict__ total) {
  unsigned long long s = 0;
  for (uint32_t l = blockIdx.x * blockDim.x + threadIdx.x; l < n_loc; l += gridDim.x * blockDim.x)
    s += indeg[deal_global(l, deal.P, deal.p)];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(total, s);
}
// edges of a pair -> groups of its segment (every pair of the staircase keeps at least one group, so
// that the row of a group follows from counting segment starts)
__global__ void k_cb_groups(uint32_t* __restrict__ cnt, uint64_t S) {
  for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < S; e += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = cnt[e];
    cnt[e] = c ? (c + CB_G - 1) / CB_G : 1u;
  }
}
__global__ void k_fill_u2(uint2* __restrict__ a, uint64_t count, uint2 v) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
    a[i] = v;
}
__global__ void k_cb_bits(const uint32_t* __restrict__ goff, uint64_t S, uint32_t* __restrict__ bits) {
  for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < S; e += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t g = goff[e];
    atomicOr(bits + (g >> 5), 1u << (g & 31u));
  }
}
// SELL slice widths: the longest lane of the slice, in 4-edge groups
__global__ void k_sell_widths(const uint32_t* __restrict__ lens, uint32_t n_loc, uint32_t num_slices,
                              uint32_t* __restrict__ units) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t sidx = warp; sidx < num_slices; sidx += nwarps) {
    const uint32_t l = 32 * sidx + lane;
    const uint32_t w = warp_max(l < n_loc ? lens[l] : 0u);
    if (lane == 0) units[sidx] = ((w + 3) / 4) * 32;  // uint4 entries of the slice
  }
}
__global__ void k_sell_meta(const uint32_t* __restrict__ units, const uint32_t* __restrict__ bases,
                            uint32_t num_slices, uint2* __restrict__ meta) {
  for (uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x; sidx < num_slices; sidx += gridDim.x * blockDim.x)
    meta[sidx] = make_uint2(bases[sidx], units[sidx] / 32);
}
// after the scan over the segment sizes: scatter the records left by the classification — block-local
// ids into the segments, all other sources into the row's SELL lane
__global__ void k_cb_fill(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ old_of,
                          const uint2* __restrict__ rec, const uint32_t* __restrict__ poff, uint32_t row0,
                          uint32_t n_cb, PrDeal deal, const uint32_t* __restrict__ goff, uint16_t* __restrict__ ids,
                          const uint2* __restrict__ slice_meta, uint32_t* __restrict__ sell) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t l = row0 + warp; l < n_cb; l += nwarps) {
    const uint32_t old = old_of[deal_global(l, deal.P, deal.p)];
    const uint32_t b0 = in_off[old], d = in_off[old + 1] - b0;
    const uint2 meta = slice_meta[l >> 5];
    for (uint32_t i = 0; i < d; i += 32 * CB_ILP) {
      uint2 r[CB_ILP];
      uint32_t g0[CB_ILP];
#pragma unroll
      for (uint32_t u = 0; u < CB_ILP; ++u) {
        const uint32_t k = i + 32 * u + lane;
        r[u] = k < d ? rec[b0 + k] : make_uint2(0u, 0xFFFFFFFFu);
      }
#pragma unroll
      for (uint32_t u = 0; u < CB_ILP; ++u)
        g0[u] = (r[u].y != 0xFFFFFFFFu && (r[u].y & CB_REC_SEG)) ? goff[poff[r[u].x >> 16] + l] : 0u;
#pragma unroll
      for (uint32_t u = 0; u < CB_ILP; ++u) {
        if (r[u].y == 0xFFFFFFFFu) continue;
        if (r[u].y & CB_REC_SEG) {
          ids[(uint64_t)g0[u] * CB_G + (r[u].y & ~CB_REC_SEG)] = (uint16_t)(r[u].x & 0xFFFFu);
        } else {
          const uint32_t q = r[u].y;
          sell[((uint64_t)meta.x + (uint64_t)(q / 4) * 32 + (l & 31u)) * 4 + (q % 4)] = r[u].x;
        }
      }
    }
  }
}
// rows without segments: the whole row goes to its SELL lane (one lane per row)
__global__ void k_sell_fill_tail(const uint32_t* __restrict__ in_off, const uint32_t* __restrict__ in_tgt,
                                 const uint32_t* __restrict__ old_of, const uint32_t* __restrict__ new_id,
                                 uint32_t n_cb, uint32_t n_loc, PrDeal deal, uint32_t num_slices,
                                 const uint2* __restrict__ meta, uint4* __restrict__ sell) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t sidx = n_cb / 32 + warp; sidx < num_slices; sidx += nwarps) {
    const uint2 m = meta[sidx];
    const uint32_t l = 32 * sidx + lane;
    if (l < n_cb) continue;  // filled by k_cb_fill (lanes of the boundary slice)
    uint32_t b = 0, d = 0;
    if (l < n_loc) {
      const uint32_t old = old_of[deal_global(l, deal.P, deal.p)];
      b = in_off[old];
      d = in_off[old + 1] - b;
    }
    for (uint32_t q = 0; q * 4 < d; ++q) {
      uint4 v = make_uint4(~0u, ~0u, ~0u, ~0u);
      const uint32_t j = 4 * q;
      if (j + 0 < d) v.x = new_id[in_tgt[b + j + 0]];
      if (j + 1 < d) v.y = new_id[in_tgt[b + j + 1]];
      if (j + 2 < d) v.z = new_id[in_tgt[b + j + 2]];
      if (j + 3 < d) v.w = new_id[in_tgt[b + j + 3]];
      sell[m.x + q * 32 + lane] = v;
    }
  }
}
__global__ void k_gather_u32(const uint32_t* __restrict__ src, const uint32_t* __restrict__ idx, uint32_t count,
                             uint32_t* __restrict__ dst) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) dst[i] = src[idx[i]];
}

// Chunks: block j's stream [gbeg[j], gbeg[j+1]) is cut every C_j groups; a cut inside a segment moves to
// the segment's end unless the segment is longer than C_j groups, in which case the cut stays and both
// neighbours handle a PART of it (side buffer + fixup), so no warp ever owns more than 2 C_j groups.
// C_j shrinks for thin blocks so that every block's stream is spread over all warps of a CTA (a lone
// warp runs at its dependency latency, ~10x below the SM's throughput).
struct CbCut {
  uint32_t pos, row;
  bool mid;
};
__device__ __forceinline__ CbCut cb_cut(const uint32_t* __restrict__ goff_j, uint32_t nr, uint32_t gend, uint32_t q,
                                        uint32_t C) {
  if (q >= gend) return CbCut{gend, nr, false};
  uint32_t lo = 0, hi = nr;  // largest row with goff_j[row] <= q
  while (hi - lo > 1) {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (goff_j[mid] <= q) lo = mid;
    else hi = mid;
  }
  const uint32_t s0 = goff_j[lo], s1 = (lo + 1 < nr) ? goff_j[lo + 1] : gend;
  if (s0 == q) return CbCut{q, lo, false};
  if (s1 - s0 > C) return CbCut{q, lo, true};
  return CbCut{s1, lo + 1, false};
}
__global__ void k_cb_chunks(const uint32_t* __restrict__ goff, const uint32_t* __restrict__ poff,
                            const uint32_t* __restrict__ nrows, const uint32_t* __restrict__ gbeg,
                            const uint32_t* __restrict__ cfirst, const uint32_t* __restrict__ cgrp, uint32_t KB,
                            uint32_t n_chunks, uint4* __restrict__ chunks, uint32_t* __restrict__ tail_slot,
                            uint32_t* __restrict__ fix_list, uint32_t* __restrict__ n_fix /* [1] = largest cut row */) {
  for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < n_chunks; c += gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = KB;  // block with cfirst[j] <= c < cfirst[j + 1]
    while (hi - lo > 1) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (cfirst[mid] <= c) lo = mid;
      else hi = mid;
    }
    const uint32_t j = lo, k = c - cfirst[j];
    const uint32_t C = cgrp[j];  // groups per chunk in this block (thin blocks use small chunks)
    const uint32_t* goff_j = goff + poff[j];
    const uint32_t nr = nrows[j], g0 = gbeg[j], g1 = gbeg[j + 1];
    const bool last = c + 1 == cfirst[j + 1];
    const CbCut a = cb_cut(goff_j, nr, g1, g0 + k * C, C);
    const CbCut b = last ? CbCut{g1, nr, false} : cb_cut(goff_j, nr, g1, g0 + (k + 1) * C, C);
    uint32_t fl = 0;
    if (a.mid) fl |= CB_HEAD_CONT;
    if (b.mid) fl |= CB_TAIL_CONT;
    const uint32_t last_row = b.mid ? b.row : b.row - 1;  // row of the chunk's last group
    if (a.mid && last_row == a.row) fl |= CB_INTERIOR;
    const uint32_t row_before = a.mid ? a.row : a.row - 1;
    chunks[c] = make_uint4(a.pos, b.pos, row_before, j | (fl << 24));
    tail_slot[c] = b.mid ? poff[j] + b.row : CB_NONE;
    if (b.mid && !(fl & CB_INTERIOR)) {
      fix_list[atomicAdd(n_fix, 1u)] = c;
      atomicMax(n_fix + 1, b.row);
    }
  }
}

// ---- sweep kernels (JACOBI) ------------------------------------------------------------------
struct PrArgs {
  const uint32_t* outdeg;
  const float* x_cur;
  float* x_next;
  float* mc_next;       // multicast mapping of x_next on every rank (NULL: unicast peer stores)
  float* peer_next[7];  // peer-mapped copies of x_next (fused allgather over NVLink); n_peers used
  uint32_t n_peers;
  uint32_t n;
  float* scores;
  PrDeal deal;
  uint32_t n_loc, n_cb;
  uint32_t n_fin_warp;  // rows [0, n_fin_warp) own segments in many blocks (finish: one CTA per 32 rows)
  uint32_t fin_hub_ctas;  // finish: CTAs [0, fin_hub_ctas) take those groups, the rest the other rows
  uint32_t n_fin;       // rows [0, n_fin) are completed by k_pr_finish (rem[] + partials); rows [n_fin, n_cb) own
                        // segments in at most SELL_FEW blocks and are completed by their k_pr_sell lane
  uint32_t few_kb, few_nrows[SELL_FEW], few_poff[SELL_FEW];  // the first blocks' row prefixes / partial offsets
  uint32_t fix_in_sell; // k_pr_sell adds the parts of cut segments first (no k_pr_fixup launch)
  const uint32_t* fin_kb;  // [ceil(n_cb / 32)] blocks in which the first row of each 32-row group owns a segment
  // column blocks
  uint32_t B, KB;
  const uint32_t* blk;
  const uint32_t* nrows;
  const uint32_t* poff;
  const uint2* cb_ids;
  const uint32_t* cb_bits;
  float* partial;
  const uint4* chunks;
  uint32_t n_chunks;
  const uint32_t* tail_slot;
  double* side;
  const uint32_t* fix_list;
  uint32_t n_fix;
  const uint2* tasks;
  uint32_t n_tasks, n_task_ranges;
  uint32_t* task_ctr;
  float* rem;
  // SELL rows
  const uint4* sell;
  const uint2* slice_meta;
  uint32_t num_slices;
  // error / stop rule
  double* block_err;
  double* err_hist;
  uint32_t* ctrl;
  uint32_t err_base_fin;  // block_err slots [0, err_base_fin) belong to the SELL CTAs
  float base, damping;
  double tolerance;
  double extra_err;   // closed-form error of the skipped zero-in-degree rows (first sweep only)
  uint32_t sweep;     // index inside the current batch
  uint32_t sweep_no;  // 1-based global sweep number
};

// 8 gathers per lane in straight-line predicated code (padding id ~0 reads nothing).  Measured in round 1
// (profiles/r01_sweep_hot_head.txt): per-target if/else made every load wait for a scoreboard slot of
// the previous one, and every pending miss holds an L1 line — so this kernel uses NO shared memory at
// all and leaves the whole 228 KB to L1 (a 128 KB shared-memory mirror of the hottest sources was
// slower than two mirror-less CTAs per SM: profiles/r02_sweep_breakdown.txt).
__device__ __forceinline__ void pr_gather(const float* x, const uint4& ta, const uint4& tb, float (&v)[8]) {
  const uint32_t t[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %1, 0xffffffff;\n\t"
        "mov.f32 %0, 0f00000000;\n\t"
        "@p ld.global.nc.f32 %0, [%2];\n\t}"
        : "=f"(v[j])
        : "r"(t[j]), "l"(x + t[j]));
  }
}
__device__ __forceinline__ float pr_sum8(const float (&v)[8]) {
  return ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
}
__device__ __forceinline__ uint4 pr_ld4(const uint4* p) { return ld_stream_u4(reinterpret_cast<const uint32_t*>(p)); }

// the per-vertex update of page_rank.rs:148-158 with the reference's rounding sequence; gr = global row
template <bool PEERS>
__device__ __forceinline__ double pr_update(uint32_t gr, float sum, float old, uint32_t deg, const PrArgs& a) {
  const float nw = __fadd_rn(a.base, __fmul_rn(a.damping, sum));
  a.scores[gr] = nw;
  const float xo = __fdiv_rn(nw, (float)deg);
  if (PEERS && a.mc_next) {
    // one store, replicated by the NVSwitch into every rank's next vector (this rank's included)
    asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(a.mc_next + gr), "f"(xo) : "memory");
  } else {
    a.x_next[gr] = xo;
    if (PEERS)
      for (uint32_t p = 0; p < a.n_peers; ++p) a.peer_next[p][gr] = xo;
  }
  return fabs((double)__fsub_rn(nw, old));
}

// ---- column blocks ------------------------------------------------------------------------------------
// One warp, one chunk: groups [g0, g1) of block j's stream, 64 groups (256 ids) per step.  Lane L owns
// the ADJACENT groups 2L and 2L+1 of the even-aligned window (one 128-bit load).  Inside a lane the two
// group sums are combined when they belong to the same row; across lanes the value of the run that is
// open at the end of each lane goes through a segmented inclusive scan (5 shuffles per 256 ids); a run
// that spans steps is carried in f64.  The row of a group follows from counting segment-start bits.
// A lane ends at most two runs per step: the one its first group closes and the one open at its end.
// SPECIAL = the chunk starts or ends inside a segment (rare: segments longer than a chunk); the common
// instantiation carries none of the side-buffer logic.
template <bool SPECIAL>
__device__ __forceinline__ void cb_emit(const PrArgs& a, uint32_t c, bool is_end, uint32_t q, uint32_t last,
                                        bool run_continues, bool last_step, bool tail_cont, bool in_head,
                                        uint32_t cum, uint32_t slot0, double tot) {
  if (!is_end) return;
  if (SPECIAL) {
    if (q == last && run_continues && !last_step) return;  // carried into the next step
    if (in_head && cum == 0) a.side[2 * (size_t)c] = tot;                        // tail part of a cut segment
    else if (q == last && last_step && tail_cont) a.side[2 * (size_t)c + 1] = tot;  // head part of one
    else a.partial[slot0 + cum] = (float)tot;
  } else {
    if (q == last && run_continues) return;  // carried into the next step
    a.partial[slot0 + cum] = (float)tot;
  }
}
template <bool SPECIAL>
__device__ __forceinline__ void cb_chunk_impl(const PrArgs& a, const float* xs, uint32_t c, const uint4 ch,
                                              uint32_t lane, uint32_t pad2) {
  const uint32_t g0 = ch.x, g1 = ch.y;
  const uint32_t j = ch.w & 0xFFFFFFu, fl = ch.w >> 24;
  const bool head_cont = SPECIAL && (fl & CB_HEAD_CONT), tail_cont = SPECIAL && (fl & CB_TAIL_CONT);
  uint32_t slot0 = a.poff[j] + ch.z;  // staircase slot of the row "before" the first segment start
  bool in_head = head_cont;
  double carry = 0.0;
  const uint32_t le_mask = 0xFFFFFFFFu >> (31u - lane);
  const uint32_t ia = 2 * lane, ib = ia + 1;
  const uint4* ids16 = reinterpret_cast<const uint4*>(a.cb_ids);  // pairs of groups
  const uint4 padv = make_uint4(pad2, pad2, pad2, pad2);
  const uint32_t gs0 = g0 & ~1u;
  uint4 ids = padv;
  if (gs0 + ia < g1) ids = ld_stream_u4(reinterpret_cast<const uint32_t*>(ids16 + (gs0 >> 1) + lane));
  for (uint32_t gs = gs0; gs < g1; gs += 64) {
    uint4 nids = padv;
    if (gs + 64 + ia < g1) nids = ld_stream_u4(reinterpret_cast<const uint32_t*>(ids16 + ((gs + 64) >> 1) + lane));
    // groups outside [g0, g1) belong to the neighbouring chunks
    if (gs + ia < g0) ids.x = ids.y = pad2;
    if (gs + ib >= g1) ids.z = ids.w = pad2;
    const uint32_t wi = gs >> 5, sh = gs & 31u;
    const uint32_t w0 = __ldg(a.cb_bits + wi), w1 = __ldg(a.cb_bits + wi + 1), w2 = __ldg(a.cb_bits + wi + 2);
    unsigned long long W = ((unsigned long long)__funnelshift_r(w1, w2, sh) << 32) | __funnelshift_r(w0, w1, sh);
    const uint32_t nvalid = min(64u, g1 - gs);
    if (nvalid < 64) W &= (1ull << nvalid) - 1ull;
    if (gs < g0) W &= ~1ull;
    const uint32_t last = nvalid - 1;
    const bool last_step = gs + 64 >= g1;
    // does the run of the last valid group go on after this step (inside the chunk / past its end)?
    const bool run_continues = last_step ? tail_cont : !((w2 >> sh) & 1u);
    const float va = xs[ids.x & 0xFFFFu] + xs[ids.x >> 16] + (xs[ids.y & 0xFFFFu] + xs[ids.y >> 16]);
    const float vb = xs[ids.z & 0xFFFFu] + xs[ids.z >> 16] + (xs[ids.w & 0xFFFFu] + xs[ids.w >> 16]);
    const uint32_t pair = (uint32_t)(W >> ia) & 3u;
    const bool fa = pair & 1u, fb = pair & 2u;
    float incl = fb ? vb : va + vb;  // this lane's share of the run open at its end
    const uint32_t below = __ballot_sync(0xFFFFFFFFu, pair != 0) & le_mask;
    const int seg_start = below ? 31 - __clz(below) : -1;
    const int lo = seg_start < 0 ? 0 : seg_start;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if ((int)lane - d >= lo) incl += t;
    }
    const double incl_d = (double)incl + (seg_start < 0 ? carry : 0.0);
    double x_in = __shfl_up_sync(0xFFFFFFFFu, incl_d, 1);  // the run open at the end of the previous lane
    if (lane == 0) x_in = carry;
    const uint32_t cum_a = __popcll(W & ((2ull << ia) - 1ull));  // segment starts at positions <= ia
    const uint32_t cum_b = cum_a + (fb ? 1u : 0u);
    const bool valid_a = gs + ia >= g0 && ia <= last, valid_b = ib <= last;
    const bool nxt = ib < 63 ? ((W >> (ib + 1)) & 1ull) != 0 : false;
    cb_emit<SPECIAL>(a, c, valid_a && (ia == last || fb), ia, last, run_continues, last_step, tail_cont, in_head,
                     cum_a, slot0, (fa ? 0.0 : x_in) + (double)va);
    cb_emit<SPECIAL>(a, c, valid_b && (ib == last || nxt), ib, last, run_continues, last_step, tail_cont, in_head,
                     cum_b, slot0, incl_d);
    const double tl = __shfl_sync(0xFFFFFFFFu, incl_d, 31);
    carry = (run_continues && !last_step) ? tl : 0.0;
    if (SPECIAL && W) in_head = false;
    slot0 += __popcll(W);
    ids = nids;
  }
}
__device__ __forceinline__ void cb_chunk(const PrArgs& a, const float* xs, uint32_t c, uint32_t lane, uint32_t pad2) {
  const uint4 ch = a.chunks[c];
  if (ch.x >= ch.y) return;
  if ((ch.w >> 24) & (CB_HEAD_CONT | CB_TAIL_CONT)) cb_chunk_impl<true>(a, xs, c, ch, lane, pad2);
  else cb_chunk_impl<false>(a, xs, c, ch, lane, pad2);
}

// ---- TMA bulk copy of a source block into shared memory (cp.async.bulk + mbarrier) -----------------
// One thread asks the copy engine for the block's 192 KB and every thread waits on the mbarrier's phase:
// no load/store instruction of the CTA is spent on the transfer and it runs at the SM's L2 bandwidth
// (the LDG.128 -> STS.128 loop it replaces kept one 16 KB wave in flight: 12 round trips per block).
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(arrivals) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(mbar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(mbar)
               : "memory");
}

// Persistent CTAs pull TASKS (32 consecutive chunks of one block).  The task list (fattest blocks first)
// is split into one contiguous RANGE per CTA, each with its own atomic cursor: a CTA first drains its own
// range — consecutive tasks of one block, so the 192 KB block is loaded once, not once per task — and then
// steals from the other ranges' cursors.  Self-balancing whatever else shares the SM and however uneven the
// thin blocks are (a purely static split ran 2.4x slower, one global cursor reloads the block for every
// task: profiles/r02_sweep_breakdown.txt).  Claiming the next task one task ahead (to hide the atomic's
// round trip) was measured and dropped: a claimed task cannot be stolen, which costs more at the tail.
__global__ void __launch_bounds__(PR_THREADS, 1) k_pr_cb(const PrArgs a) {
  extern __shared__ __align__(128) float smem[];
  float* xs = smem;  // B entries of x_cur + one zero slot (the pad id)
  __shared__ uint32_t s_task, s_next;
  __shared__ __align__(8) unsigned long long s_mbar;
  if (a.ctrl[0] != 0) return;  // tolerance already met by an earlier sweep of this batch
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t B = a.B;
  const uint32_t pad2 = B | (B << 16);
  const uint32_t R = gridDim.x;  // ranges = CTAs
  const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar);
  const uint32_t xs_smem = (uint32_t)__cvta_generic_to_shared(xs);
  const bool bulk_ok = (reinterpret_cast<uintptr_t>(a.x_cur) & 15u) == 0;  // cp.async.bulk moves 16-byte units
  uint32_t phase = 0;
  if (threadIdx.x == 0) mbar_init(mbar, 1);
  if (threadIdx.x < 4) xs[B + threadIdx.x] = 0.0f;  // the pad id's zero slot: never overwritten
  uint32_t cur_j = CB_NONE;
  uint32_t r = blockIdx.x;  // range being drained (warp 0 keeps it)
  __syncthreads();  // mbarrier + zero slot are set up
  for (;;) {
    if (warp == 0) {
      uint32_t t = CB_NONE;
      for (;;) {
        const uint32_t lo = (uint32_t)((uint64_t)a.n_tasks * r / R), hi = (uint32_t)((uint64_t)a.n_tasks * (r + 1) / R);
        uint32_t k = CB_NONE;
        if (lane == 0) {
          k = lo + atomicAdd(a.task_ctr + r, 1u);
          if (k >= hi) k = CB_NONE;
        }
        t = __shfl_sync(0xFFFFFFFFu, k, 0);
        if (t != CB_NONE) break;
        // this range is drained: the lanes probe the other ranges' cursors 32 at a time (plain loads)
        uint32_t found = CB_NONE;
        for (uint32_t base = 1; base < R && found == CB_NONE; base += 32) {
          uint32_t q = r + base + lane;
          if (q >= R) q -= R;
          bool ok = false;
          if (base + lane < R) {
            const uint32_t qlo = (uint32_t)((uint64_t)a.n_tasks * q / R), qhi = (uint32_t)((uint64_t)a.n_tasks * (q + 1) / R);
            ok = *((volatile uint32_t*)(a.task_ctr + q)) < qhi - qlo;
          }
          const uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
          if (m) found = __shfl_sync(0xFFFFFFFFu, q, __ffs(m) - 1);
        }
        if (found == CB_NONE) break;  // every range is drained
        r = found;
      }
      if (lane == 0) s_task = t;
    }
    __syncthreads();  // also: every warp is done with the previous task's block
    const uint32_t t = s_task;
    if (threadIdx.x == 0) s_next = PR_WARPS;  // every warp is past its last claim of the previous task
    __syncthreads();
    if (t == CB_NONE) break;
    const uint2 task = a.tasks[t];  // (first chunk, chunk count | block rank << 8)
    const uint32_t j = task.y >> 8;
    if (j != cur_j) {
      const uint64_t x0 = (uint64_t)a.blk[j] * B;
      const uint32_t cnt = (uint32_t)min((uint64_t)B, (uint64_t)a.n - x0);
      if (bulk_ok) {
        const uint32_t bulk = cnt & ~3u;
        if (threadIdx.x == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the block's old contents were read through the generic proxy
          mbar_expect_tx(mbar, bulk * 4u);
          for (uint32_t off = 0; off < bulk; off += 4096u)  // 16 KB pieces
            bulk_g2s(xs_smem + off * 4u, a.x_cur + x0 + off, min(4096u, bulk - off) * 4u, mbar);
        }
        if (threadIdx.x >= 32 && threadIdx.x - 32 < cnt - bulk) xs[bulk + threadIdx.x - 32] = a.x_cur[x0 + bulk + threadIdx.x - 32];
        mbar_wait(mbar, phase);
        phase ^= 1u;
      } else {
        for (uint32_t i = threadIdx.x; i < cnt; i += PR_THREADS) xs[i] = a.x_cur[x0 + i];
      }
      cur_j = j;
      __syncthreads();
    }
    // a warp starts with chunk `warp` of the task and claims further ones from the CTA's counter
    const uint32_t nchunks = task.y & 0xFFu;
    for (uint32_t k = warp; k < nchunks;) {
      cb_chunk(a, xs, task.x + k, lane, pad2);
      uint32_t nx = 0;
      if (lane == 0) nx = atomicAdd(&s_next, 1u);
      k = __shfl_sync(0xFFFFFFFFu, nx, 0);
    }
  }
}

// Segments cut by chunk boundaries (segments longer than a chunk): one warp per segment adds its parts
// in a fixed order — the head part of the first chunk, then lanes over the following chunks (a fixed
// xor tree per batch of 32).  Tiny; runs after k_pr_cb (as k_pr_fixup, or as the prologue of k_pr_sell).
__device__ __forceinline__ void cb_fix_segment(const PrArgs& a, uint32_t c0, uint32_t lane) {
  double t = a.side[2 * (size_t)c0 + 1];
  for (uint32_t k0 = c0 + 1;; k0 += 32) {
    const uint32_t k = k0 + lane;
    // the walk ends at the first chunk that is not entirely inside the segment (sentinel chunk after the last)
    const uint32_t fl = a.chunks[min(k, a.n_chunks)].w >> 24;
    const bool inside = k < a.n_chunks && (fl & CB_INTERIOR) && (fl & CB_TAIL_CONT);
    const uint32_t stop = __ballot_sync(0xFFFFFFFFu, !inside);
    const uint32_t upto = stop ? (uint32_t)__ffs(stop) - 1 : 31u;  // last lane that contributes
    t += warp_sum(lane <= upto ? a.side[2 * (size_t)k] : 0.0);
    if (stop) break;
  }
  if (lane == 0) a.partial[a.tail_slot[c0]] = (float)t;
}
__global__ void k_pr_fixup(const PrArgs a) {
  if (a.ctrl[0] != 0) return;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t i = gw; i < a.n_fix; i += nw) cb_fix_segment(a, a.fix_list[i], lane);
}

// ---- SELL-32 sweep: one lane per row ------------------------------------------------------------
// A lane reads its row four targets at a time (128-bit, coalesced: the slice is stored group-major,
// lane-minor), gathers, and adds in row order.  The next slice's first targets and row metadata are
// requested while the current slice is processed.  Rows below n_cb only hold the edges that are not in
// a column-block segment: their sum goes to rem[] and the finish kernel completes them.
// The kernel needs no shared memory: two 512-thread CTAs per SM.
template <bool PEERS>
__global__ void __launch_bounds__(PR_SELL_THREADS, 2) k_pr_sell(const PrArgs a) {
  constexpr int NT = PR_SELL_THREADS;
  constexpr int NW = NT / 32;
  __shared__ double warp_err[NW];
  if (a.ctrl[0] != 0) return;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (a.fix_in_sell) {
    // segments cut by chunk boundaries (hub rows only: they are completed by k_pr_finish, after this kernel)
    const uint32_t gw0 = blockIdx.x * NW + warp, nw0 = gridDim.x * NW;
    for (uint32_t i = gw0; i < a.n_fix; i += nw0) cb_fix_segment(a, a.fix_list[i], lane);
  }
  const float* __restrict__ x = a.x_cur;
  double err = 0.0;
  const uint32_t stride = gridDim.x * NW;
  const uint4 pad = make_uint4(~0u, ~0u, ~0u, ~0u);
  const uint32_t P = a.deal.P, pp = a.deal.p;
  // slices are dealt CTA-minor: the widest slices (the first ones) land on different SMs, not on the 16
  // warps of CTA 0 (an eighth-shard ran with its busiest SM 31 % above the average otherwise)
  uint32_t sidx = warp * gridDim.x + blockIdx.x;
  // pipeline state: metadata of this and the next slice, first two target groups + row data of this one
  uint2 meta = make_uint2(0, 0), nmeta = meta;
  uint4 ta = pad, tb = pad;
  float old = 0.0f;
  uint32_t deg = 1;
  if (sidx < a.num_slices) {
    meta = __ldg(a.slice_meta + sidx);
    if (sidx + stride < a.num_slices) nmeta = __ldg(a.slice_meta + sidx + stride);
    const uint4* base = a.sell + meta.x + lane;
    if (0 < meta.y) ta = pr_ld4(base);
    if (1 < meta.y) tb = pr_ld4(base + 32);
    const uint32_t l = 32 * sidx + lane;
    if (l >= a.n_fin && l < a.n_loc) {
      const uint32_t gr = deal_global(l, P, pp);
      old = a.scores[gr];
      deg = a.outdeg[gr];
    }
  }
  while (sidx < a.num_slices) {
    const uint32_t w4 = meta.y;
    const uint4* base = a.sell + meta.x + lane;
    const uint32_t l = 32 * sidx + lane;
    // next slice: first groups, row data; metadata of the slice after it
    const uint32_t nidx = sidx + stride;
    uint4 nta = pad, ntb = pad;
    float nold = 0.0f;
    uint32_t ndeg = 1;
    uint2 nnmeta = make_uint2(0, 0);
    if (nidx < a.num_slices) {
      const uint4* nbase = a.sell + nmeta.x + lane;
      if (0 < nmeta.y) nta = pr_ld4(nbase);
      if (1 < nmeta.y) ntb = pr_ld4(nbase + 32);
      const uint32_t nl = 32 * nidx + lane;
      if (nl >= a.n_fin && nl < a.n_loc) {
        const uint32_t ngr = deal_global(nl, P, pp);
        nold = a.scores[ngr];
        ndeg = a.outdeg[ngr];
      }
      if (nidx + stride < a.num_slices) nnmeta = __ldg(a.slice_meta + nidx + stride);
    }
    // a row with segments in at most SELL_FEW blocks is completed here: its partials (written by k_pr_cb,
    // which ran before) are requested now and added after the gathers, in block order like k_pr_finish
    float part[SELL_FEW];
#pragma unroll
    for (uint32_t j = 0; j < SELL_FEW; ++j) {
      part[j] = 0.0f;
      if (l >= a.n_fin && j < a.few_kb && l < a.few_nrows[j]) part[j] = a.partial[(size_t)a.few_poff[j] + l];
    }
    float acc = 0.0f;
    for (uint32_t q = 0; q < w4; q += 2) {
      // targets of the next two groups are requested before this group's gathers are consumed
      const uint4 na = (q + 2 < w4) ? pr_ld4(base + (q + 2) * 32) : pad;
      const uint4 nb = (q + 3 < w4) ? pr_ld4(base + (q + 3) * 32) : pad;
      float v[8];
      pr_gather(x, ta, tb, v);
      acc += pr_sum8(v);
      ta = na;
      tb = nb;
    }
    if (l < a.n_fin) {
      a.rem[l] = acc;
    } else if (l < a.n_loc) {
      if (l < a.n_cb) {
        double sum = (double)acc;
#pragma unroll
        for (uint32_t j = 0; j < SELL_FEW; ++j)
          if (j < a.few_kb && l < a.few_nrows[j]) sum += (double)part[j];
        acc = (float)sum;
      }
      err += pr_update<PEERS>(deal_global(l, P, pp), acc, old, deg, a);
    }
    sidx = nidx;
    meta = nmeta;
    nmeta = nnmeta;
    ta = nta;
    tb = ntb;
    old = nold;
    deg = ndeg;
  }
  err = warp_sum(err);
  if (lane == 0) warp_err[warp] = err;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tt = 0.0;
#pragma unroll
    for (int w = 0; w < NW; ++w) tt += warp_err[w];
    a.block_err[blockIdx.x] = tt;
  }
}

// ---- finish: rows with segments = partials of their blocks (fixed order, f64) + SELL remainder -----
// 32-row groups that own segments in more than FIN_CTA_BLOCKS blocks (the hubs: a prefix) get a CTA
// each; all other rows one lane each (coalesced across the warp's 32 rows).  The last CTA to
// finish reduces all CTA error partials in a fixed order and evaluates the stop rule of
// page_rank.rs:107 on the device.
__host__ __device__ __forceinline__ uint32_t fin_blocks_of(const uint32_t* __restrict__ nrows, uint32_t KB, uint32_t l) {
  uint32_t lo = 0, hi = KB;  // first j with nrows[j] <= l  (nrows is non-increasing)
  while (lo < hi) {
    const uint32_t mid = (lo + hi) / 2;
    if (nrows[mid] > l) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
// FIN_U = 32-row groups per warp iteration of the rows that are not hub groups: 2 (and 16 blocks' partials
// in flight) when every warp has a single iteration to do — the walk is a latency chain, fewer rounds win;
// 4 (4 blocks in flight) when the grid is capped and the kernel is throughput bound (RMAT-26 on one GPU).
template <bool PEERS, uint32_t FIN_U>
__global__ void __launch_bounds__(PR_FIN_THREADS) k_pr_finish(const PrArgs a) {
  constexpr int FIN_WARPS = PR_FIN_THREADS / 32;
  __shared__ double warp_err[FIN_WARPS];
  __shared__ bool is_last;
  if (a.ctrl[0] != 0) return;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double err = 0.0;
  const uint32_t P = a.deal.P, pp = a.deal.p;
  if (blockIdx.x == 0)  // next sweep's column-block task cursors
    for (uint32_t i = threadIdx.x; i < a.n_task_ranges; i += PR_FIN_THREADS) a.task_ctr[i] = 0;
  // hub rows (segments in more than FIN_CTA_BLOCKS blocks): one CTA per 32-row group — lane = row,
  // warp w adds blocks w, w + 8, ... (independent coalesced loads), warp 0 adds the 8 sums in order
  __shared__ double part[FIN_WARPS][32];
  // fin_hub_ctas != 0: CTAs [0, fin_hub_ctas) take the hub groups, the others the remaining rows
  const bool split = a.fin_hub_ctas != 0;  // else every CTA does both parts
  const uint32_t H = split ? a.fin_hub_ctas : gridDim.x, T0 = split ? a.fin_hub_ctas : 0u;
  for (uint32_t g = blockIdx.x; blockIdx.x < H && g * 32 < a.n_fin_warp; g += H) {
    const uint32_t l = g * 32 + lane;
    const uint32_t kb = __ldg(a.fin_kb + g);  // blocks of the group's first row (it has the most)
    double s = 0.0;
#pragma unroll 8
    for (uint32_t j = warp; j < kb; j += FIN_WARPS)
      if (l < __ldg(a.nrows + j)) s += (double)a.partial[(size_t)__ldg(a.poff + j) + l];
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && l < a.n_fin) {
      double t = (double)a.rem[l];
#pragma unroll
      for (int w = 0; w < FIN_WARPS; ++w) t += part[w][lane];
      const uint32_t gr = deal_global(l, P, pp);
      err += pr_update<PEERS>(gr, (float)t, a.scores[gr], a.outdeg[gr], a);
    }
    __syncthreads();
  }
  // all other rows with segments: one lane per row, FIN_U consecutive 32-row groups per warp iteration,
  // 16 blocks' partials requested at a time (the walk is latency bound, not bandwidth bound: rounds count)
  const uint32_t tail_groups = (a.n_fin - a.n_fin_warp + 31) / 32;
  const uint32_t tw = (blockIdx.x - T0) * FIN_WARPS + warp, tnw = (gridDim.x - T0) * FIN_WARPS;
  for (uint32_t w = tw * FIN_U; blockIdx.x >= T0 && w < tail_groups; w += tnw * FIN_U) {
    const uint32_t l0 = a.n_fin_warp + 32 * w;
    const uint32_t kb = __ldg(a.fin_kb + (l0 >> 5));  // blocks of the first row (it has the most)
    uint32_t l[FIN_U], gr[FIN_U], deg[FIN_U];
    float old[FIN_U];
    double s[FIN_U];
#pragma unroll
    for (uint32_t u = 0; u < FIN_U; ++u) {
      l[u] = l0 + 32 * u + lane;
      gr[u] = 0;
      deg[u] = 1;
      old[u] = 0.0f;
      s[u] = 0.0;
      if (l[u] < a.n_fin) {
        gr[u] = deal_global(l[u], P, pp);
        old[u] = a.scores[gr[u]];
        deg[u] = a.outdeg[gr[u]];
        s[u] = (double)a.rem[l[u]];
      }
    }
#pragma unroll(FIN_U == 2 ? 16 : 4)
    for (uint32_t j = 0; j < kb; ++j) {
      const uint32_t nr = __ldg(a.nrows + j);
      const float* __restrict__ pj = a.partial + __ldg(a.poff + j);
#pragma unroll
      for (uint32_t u = 0; u < FIN_U; ++u)
        if (l[u] < nr) s[u] += (double)pj[l[u]];
    }
#pragma unroll
    for (uint32_t u = 0; u < FIN_U; ++u)
      if (l[u] < a.n_fin) err += pr_update<PEERS>(gr[u], (float)s[u], old[u], deg[u], a);
  }
  err = warp_sum(err);
  if (lane == 0) warp_err[warp] = err;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < FIN_WARPS; ++w) t += warp_err[w];
    a.block_err[a.err_base_fin + blockIdx.x] = t;
    __threadfence();
    unsigned ticket = atomicAdd(&a.ctrl[1], 1u);
    is_last = (ticket == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // fixed-order reduction of all CTA partials (deterministic error)
  const uint32_t total = a.err_base_fin + gridDim.x;
  double t = 0.0;
  for (uint32_t i = threadIdx.x; i < total; i += PR_FIN_THREADS) t += ((volatile double*)a.block_err)[i];
  t = warp_sum(t);
  if (lane == 0) warp_err[warp] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    double e = a.extra_err;
#pragma unroll
    for (int w = 0; w < FIN_WARPS; ++w) e += warp_err[w];
    a.err_hist[a.sweep] = e;
    a.ctrl[1] = 0;
    if (e < a.tolerance) a.ctrl[0] = a.sweep_no;
  }
}

// ---- inter-sweep barrier of the sharded path, on the device -------------------------------------------
// Every rank owns a control block in peer-mapped (symmetric) memory: arrive[q] = the last sweep rank q has
// finished, errs[sweep & 1][q] = rank q's share of that sweep's error.  After its finish kernel a rank
// publishes its error share and then its arrival into EVERY rank's block (release, system scope), waits
// until all ranks have arrived at this sweep (acquire) and adds the P shares in rank order — every rank
// gets the same total, without a host round trip or a collective.  Two error banks suffice: a rank can
// be at most one sweep ahead of the slowest (it cannot pass barrier k+1 before everyone left barrier k).
struct PrSyncBlock {
  uint32_t arrive[8];
  double errs[2][8];
};
__global__ void k_pr_sync(PrSyncBlock* self, PrSyncBlock* const* peers_dev, uint32_t P, uint32_t rank,
                          uint32_t sweep_no, const double* __restrict__ local_err, double* __restrict__ total_err,
                          uint32_t slot) {
  const uint32_t q = threadIdx.x;
  const double mine = *local_err;
  __threadfence_system();  // this rank's stores of the sweep (previous kernels) before its arrival
  if (q < P) {
    PrSyncBlock* dst = (q == rank) ? self : peers_dev[q];
    volatile double* e = &dst->errs[sweep_no & 1u][rank];
    *e = mine;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(&dst->arrive[rank]), "r"(sweep_no) : "memory");
  }
  if (q < P) {
    uint32_t seen;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(&self->arrive[q]) : "memory");
    } while ((int32_t)(seen - sweep_no) < 0);
  }
  __syncthreads();
  if (q == 0) {
    double t = 0.0;
    for (uint32_t r = 0; r < P; ++r) t += ((volatile double*)self->errs[sweep_no & 1u])[r];
    total_err[slot] = t;
  }
}

// own == 0: scores of rows this rank does not own stay 0 so that the ranks' vectors can be summed
__global__ void k_pr_init(uint32_t n, uint32_t n_active, float init, float base, PrDeal deal,
                          const uint32_t* __restrict__ outdeg, float* __restrict__ x0,
                          float* __restrict__ x1, float* __restrict__ scores) {
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
    float d = (float)outdeg[r];
    x0[r] = __fdiv_rn(init, d);  // page_rank.rs:75-79; +inf for dangling vertices, never gathered
    const bool mine = ((r >> 5) % deal.P) == deal.p;
    if (r < n_active) {
      scores[r] = mine ? init : 0.0f;
    } else {
      // no in-edges: after the first sweep score == base + damping * 0 == base, for ever
      scores[r] = deal.p == 0 ? base : 0.0f;
      x1[r] = __fdiv_rn(base, d);
    }
  }
}
__global__ void k_pr_fill_inactive(uint32_t n, uint32_t n_active, float base,
                                   const uint32_t* __restrict__ outdeg, float* __restrict__ x) {
  for (uint32_t r = n_active + blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x)
    x[r] = __fdiv_rn(base, (float)outdeg[r]);
}
__global__ void k_unpermute(const float* __restrict__ src, const uint32_t* __restrict__ new_id,
                            uint32_t n, float* __restrict__ dst) {
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
    dst[v] = src[new_id[v]];
}

// ---- EXACT: the reference sweep on one warp ---------------------------------------------------
// page_rank.rs:58-168 with the loop of :142-160 executed in id order.  Lanes fetch 32 gathered values
// at a time; every lane then performs the same sequential f32 additions in CSR order.
__global__ void __launch_bounds__(32) k_pr_exact(const uint32_t* __restrict__ in_off,
                                                 const uint32_t* __restrict__ in_tgt,
                                                 const uint32_t* __restrict__ out_off, uint32_t n,
                                                 uint64_t max_iterations, double tolerance, float damping,
                                                 float* scores, float* out, uint64_t* ran,
                                                 double* error) {
  const uint32_t lane = threadIdx.x;
  const float nf = (float)n;
  const float init = __fdiv_rn(1.0f, nf);
  const float base = __fdiv_rn(__fsub_rn(1.0f, damping), nf);
  for (uint32_t v = lane; v < n; v += 32) {
    out[v] = __fdiv_rn(init, (float)(out_off[v + 1] - out_off[v]));
    scores[v] = init;
  }
  __syncwarp();
  uint64_t it = 0;
  double err = 0.0;
  for (;;) {
    err = 0.0;
    for (uint32_t u = 0; u < n; ++u) {
      const uint32_t b = in_off[u], e = in_off[u + 1];
      float tot = 0.0f;
      for (uint32_t i = b; i < e; i += 32) {
        const uint32_t cnt = min(32u, e - i);
        float val = 0.0f;
        if (lane < cnt) val = ((volatile float*)out)[in_tgt[i + lane]];
        for (uint32_t j = 0; j < cnt; ++j) tot = __fadd_rn(tot, __shfl_sync(0xFFFFFFFFu, val, j));
      }
      const float old = scores[u];
      const float nw = __fadd_rn(base, __fmul_rn(damping, tot));
      err += fabs((double)__fsub_rn(nw, old));
      __syncwarp();
      if (lane == 0) {
        scores[u] = nw;
        ((volatile float*)out)[u] = __fdiv_rn(nw, (float)(out_off[u + 1] - out_off[u]));
      }
      __syncwarp();
    }
    ++it;
    if (err < tolerance || it == max_iterations) break;  // page_rank.rs:107
  }
  if (lane == 0) {
    *ran = it;
    *error = err;
  }
}

// ---- plan ------------------------------------------------------------------------------------
template <typename T>
static gb_status scan_exclusive(cudaStream_t s, T* data, uint64_t count) {
  GB_REQUIRE(count < (1ull << 31), "scan of %llu items is too long", (unsigned long long)count);
  size_t tb = 0;
  GB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, data, data, (int)count, s));
  DevBuf<uint8_t> tmp;
  GB_TRY(tmp.alloc(tb));
  GB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, data, data, (int)count, s));
  GB_CUDA(cudaStreamSynchronize(s));
  return GB_OK;
}
template <typename T>
static gb_status upload(cudaStream_t s, DevBuf<T>* dst, const std::vector<T>& src, size_t pad = 0) {
  GB_TRY(dst->alloc(std::max<size_t>(src.size(), 1), pad));
  if (!src.empty()) GB_CUDA(cudaMemcpyAsync(dst->p, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  GB_CUDA(cudaStreamSynchronize(s));  // src may be a temporary
  return GB_OK;
}
static uint32_t env_u32(const char* name, uint32_t dflt) {
  const char* e = getenv(name);
  return e && *e ? (uint32_t)strtoul(e, nullptr, 10) : dflt;
}

static gb_status build_pr_plan(const gb_graph* g, PrDeal deal, PrPlan** out_plan) {
  cudaStream_t s = g->stream;
  const uint32_t n = g->n;
  const uint64_t m = g->in.len;
  GB_REQUIRE(deal.P >= 1 && deal.p < deal.P, "bad shard %u of %u", deal.p, deal.P);
  PrPlan* p = new (std::nothrow) PrPlan();
  if (!p) return fail(GB_ERR_OOM, "host allocation failed");
  p->n = n;
  p->m = m;
  p->deal = deal;
  // every temporary below is used on s only: releasing one waits for s, not for the device (a copy
  // stream may still be bringing in the targets, see TargetFeed)
  DevBufStreamScope scope(s);
  const TargetFeed* feed = g->feed;
  gb_status st = [&]() -> gb_status {
    int dev_sms = 148;
    GB_CUDA(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, g->device));
    // knobs (experiments; defaults are the measured optima)
    uint32_t B = env_u32("GB_PR_BLOCK", CB_BLOCK_DEFAULT);
    B = std::min<uint32_t>(std::max<uint32_t>(B & ~1023u, 1024u), CB_BLOCK_MAX);
    double tau = CB_TAU_DEFAULT;
    if (const char* e = getenv("GB_PR_TAU")) tau = atof(e);
    if (!(tau > 0.0)) tau = 1e30;  // tau <= 0 switches the column blocks off
    p->B = B;
    // 1. permutation: in-degree descending, then out-degree descending, then id
    DevBuf<uint32_t> old_of;  // internal id -> original id (plan-time only)
    DevBuf<uint32_t> indeg;   // in-degree by internal id (plan-time only)
    {
      DevBuf<uint64_t> keys, keys_alt;
      DevBuf<uint32_t> ids, ids_alt;
      GB_TRY(keys.alloc(n));
      GB_TRY(keys_alt.alloc(n));
      GB_TRY(ids.alloc(n));
      GB_TRY(ids_alt.alloc(n));
      k_perm_keys<<<grid_for(n, 256), 256, 0, s>>>(g->in.off.p, g->out.off.p, n, keys.p, ids.p);
      cub::DoubleBuffer<uint64_t> kb(keys.p, keys_alt.p);
      cub::DoubleBuffer<uint32_t> vb(ids.p, ids_alt.p);
      size_t tb = 0;
      GB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, kb, vb, (int)n, 0, 64, s));
      DevBuf<uint8_t> tmp;
      GB_TRY(tmp.alloc(tb));
      GB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, kb, vb, (int)n, 0, 64, s));
      GB_TRY(p->new_id.alloc(n));
      GB_TRY(p->outdeg.alloc(n));
      GB_TRY(indeg.alloc((size_t)n + 1));
      k_perm_scatter<<<grid_for(n, 256), 256, 0, s>>>(vb.Current(), g->out.off.p, g->in.off.p, n, p->new_id.p,
                                                     p->outdeg.p, indeg.p);
      GB_TRY(old_of.alloc(n));
      GB_CUDA(cudaMemcpyAsync(old_of.p, vb.Current(), (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
      GB_CUDA(cudaGetLastError());
      GB_CUDA(cudaStreamSynchronize(s));
    }
    // 2. active rows (a prefix of the internal order) and this rank's share of them
    DevBuf<unsigned long long> counters;  // [0] active rows, [1] local edges, [2] edges in segments, [3] fix count
    GB_TRY(counters.alloc(4));
    GB_CUDA(cudaMemsetAsync(counters.p, 0, 32, s));
    k_count_active<<<grid_for(n, 256), 256, 0, s>>>(indeg.p, n, reinterpret_cast<uint32_t*>(counters.p));
    {
      unsigned long long h = 0;
      GB_CUDA(cudaMemcpyAsync(&h, counters.p, 8, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      p->n_active = (uint32_t)h;
    }
    p->n_loc = deal_count(p->n_active, deal.P, deal.p);
    if (p->n_loc) k_loc_edges<<<grid_for(p->n_loc, 256), 256, 0, s>>>(indeg.p, p->n_loc, deal, counters.p + 1);
    // 3. hot blocks: block b carries the share e_b / m of all gathers; a row of in-degree d expects
    //    d * e_b / m edges from it, and gets a segment when that is at least tau
    const uint32_t nblk = (uint32_t)(((uint64_t)n + B - 1) / B);
    uint32_t n_mega = 0;  // local rows [0, n_mega) are long enough for the sort path of the build
    std::vector<uint32_t> h_hot(nblk, CB_NONE), h_blk, h_nrows, h_poff;
    if (p->n_loc && m) {
      DevBuf<unsigned long long> blk_edges;
      DevBuf<uint32_t> dmin, rows_ge;
      GB_TRY(blk_edges.alloc(nblk));
      GB_TRY(dmin.alloc(nblk + 1));  // + one probe: the rows long enough for the sort path of the build
      GB_TRY(rows_ge.alloc(nblk + 1));
      k_blk_edges<<<nblk, 256, 0, s>>>(p->outdeg.p, n, B, blk_edges.p);
      std::vector<unsigned long long> h_edges(nblk);
      GB_CUDA(cudaMemcpyAsync(h_edges.data(), blk_edges.p, (size_t)nblk * 8, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      std::vector<uint32_t> h_dmin(nblk + 1, 0xFFFFFFFFu);
      h_dmin[nblk] = env_u32("GB_PR_MEGA", CB_MEGA_DEG) + 1;
      for (uint32_t b = 0; b < nblk; ++b)
        if (h_edges[b]) {
          const double d = std::ceil(tau * (double)m / (double)h_edges[b]);
          h_dmin[b] = d >= 4294967295.0 ? 0xFFFFFFFFu : std::max<uint32_t>(1u, (uint32_t)d);
        }
      GB_CUDA(cudaMemcpyAsync(dmin.p, h_dmin.data(), (size_t)(nblk + 1) * 4, cudaMemcpyHostToDevice, s));
      k_rows_ge<<<grid_for(nblk + 1, 128), 128, 0, s>>>(indeg.p, p->n_active, dmin.p, nblk + 1, rows_ge.p);
      std::vector<uint32_t> h_rows(nblk + 1);
      GB_CUDA(cudaMemcpyAsync(h_rows.data(), rows_ge.p, (size_t)(nblk + 1) * 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      n_mega = deal_count(h_rows[nblk], deal.P, deal.p);
      // every block with a qualifying local row is kept, however thin: a thin block costs one block load
      // (~2 us on one SM), while its ids would otherwise lengthen the SELL lanes of the hub rows, which
      // one lane walks serially
      std::vector<uint32_t> order;
      for (uint32_t b = 0; b < nblk; ++b)
        if (h_dmin[b] != 0xFFFFFFFFu && deal_count(h_rows[b], deal.P, deal.p) != 0) order.push_back(b);
      std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
        return h_rows[x] != h_rows[y] ? h_rows[x] > h_rows[y] : x < y;
      });
      if (order.size() > CB_MAX_BLOCKS) order.resize(CB_MAX_BLOCKS);
      uint64_t S = 0;
      for (uint32_t j = 0; j < order.size(); ++j) {
        const uint32_t b = order[j];
        h_hot[b] = j;
        h_blk.push_back(b);
        h_nrows.push_back(deal_count(h_rows[b], deal.P, deal.p));
        h_poff.push_back((uint32_t)S);
        S += h_nrows.back();
        GB_REQUIRE(S < 0xFFFFFFF0ull, "column-block staircase too large (%llu pairs)", (unsigned long long)S);
      }
      h_poff.push_back((uint32_t)S);
      p->S = S;
    }
    p->KB = (uint32_t)h_blk.size();
    p->n_cb = p->KB ? h_nrows[0] : 0;
    if (h_poff.empty()) h_poff.push_back(0);
    DevBuf<uint32_t> hot_of_blk;
    GB_TRY(upload(s, &hot_of_blk, h_hot));
    GB_TRY(upload(s, &p->blk, h_blk));
    GB_TRY(upload(s, &p->nrows, h_nrows));
    GB_TRY(upload(s, &p->poff, h_poff));
    // 4. segment sizes (pairs of the staircase) and SELL lane lengths
    DevBuf<uint32_t> goff;  // [S + 1] edges per pair -> groups per pair -> first group of each pair
    DevBuf<uint32_t> lens;  // [n_loc] SELL lane lengths
    GB_TRY(goff.alloc(p->S + 1));
    GB_CUDA(cudaMemsetAsync(goff.p, 0, (p->S + 1) * 4, s));
    GB_TRY(lens.alloc(std::max<uint32_t>(p->n_loc, 1)));
    // the longest rows: key, sort, count from the sorted sequence (kept for the fill pass below)
    n_mega = std::min(n_mega, std::min(p->n_cb, (1u << (32 - CB_MEGA_JBITS)) - 1u));
    if (p->KB >= (1u << CB_MEGA_JBITS) - 1u) n_mega = 0;
    DevBuf<uint32_t> mega_keys, mega_vals, mega_start, mega_off;
    uint32_t M = 0;
    if (n_mega) {
      DevBuf<uint32_t> mdeg;
      GB_TRY(mdeg.alloc(n_mega));
      k_mega_deg<<<grid_for(n_mega, 128), 128, 0, s>>>(indeg.p, n_mega, deal, mdeg.p);
      std::vector<uint32_t> h_moff(n_mega + 1, 0);
      GB_CUDA(cudaMemcpyAsync(h_moff.data() + 1, mdeg.p, (size_t)n_mega * 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      uint64_t acc = 0;
      for (uint32_t r = 0; r < n_mega; ++r) {
        acc += h_moff[r + 1];
        if (acc >= 0xFFFFFFF0ull) {  // more mega edges than a 32-bit sort index holds: shorten the prefix
          n_mega = r;
          acc -= h_moff[r + 1];
          break;
        }
        h_moff[r + 1] = (uint32_t)acc;
      }
      h_moff.resize(n_mega + 1);
      M = n_mega ? h_moff[n_mega] : 0;
      if (M) GB_TRY(upload(s, &mega_off, h_moff));
      else n_mega = 0;
    }
    // all other rows that own segments: one record per in-edge (consumed by the fill pass)
    DevBuf<uint2> rec;
    if (p->n_cb > n_mega) {
      uint32_t dmax = 0;  // a record holds a 31-bit position
      GB_CUDA(cudaMemcpyAsync(&dmax, indeg.p + deal_global(n_mega, deal.P, deal.p), 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      GB_REQUIRE(dmax < 0x7FFFFFFFu, "a row with %u in-edges outside the sort path of the layout build", dmax);
      GB_TRY(rec.alloc(std::max<uint64_t>(m, 1)));
    }
    if (feed) {
      // the targets arrive chunk by chunk: check and classify each chunk as soon as it is there
      DevBuf<unsigned int> bad;
      GB_TRY(bad.alloc(1));
      GB_CUDA(cudaMemsetAsync(bad.p, 0, 4, s));
      for (size_t k = 0; k + 1 < feed->row_begin.size(); ++k) {
        const uint32_t v0 = feed->row_begin[k], v1 = feed->row_begin[k + 1];
        const uint64_t e0 = feed->edge_begin[k], e1 = feed->edge_begin[k + 1];
        GB_CUDA(cudaStreamWaitEvent(s, feed->ready[k], 0));
        if (e1 > e0) k_feed_check<<<grid_for(e1 - e0, 256), 256, 0, s>>>(g->in.tgt.p + e0, e1 - e0, n, bad.p);
        if (p->n_cb > n_mega && v1 > v0)
          k_cb_count_rows<<<grid_for((uint64_t)(v1 - v0), 256), 256, 0, s>>>(
              g->in.off.p, g->in.tgt.p, p->new_id.p, hot_of_blk.p, p->nrows.p, p->poff.p, p->blk.p, B, v0, v1, n, n_mega,
              p->n_cb, deal, goff.p, rec.p, lens.p, counters.p + 2);
      }
      unsigned int nbad = 0;
      GB_CUDA(cudaGetLastError());
      GB_CUDA(cudaMemcpyAsync(&nbad, bad.p, 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      GB_REQUIRE(nbad == 0, "in CSR holds %u targets >= node_count %u", nbad, n);
    } else if (p->n_cb > n_mega) {
      k_cb_count<<<grid_for((uint64_t)(p->n_cb - n_mega) * 32, 256), 256, 0, s>>>(
          g->in.off.p, g->in.tgt.p, old_of.p, p->new_id.p, hot_of_blk.p, p->nrows.p, p->poff.p, p->blk.p, B, n_mega,
          p->n_cb, deal, goff.p, rec.p, lens.p, counters.p + 2);
    }
    if (M) {
      DevBuf<uint32_t> keys_in, vals_in;
      GB_TRY(keys_in.alloc(M));
      GB_TRY(vals_in.alloc(M));
      GB_TRY(mega_keys.alloc(M));
      GB_TRY(mega_vals.alloc(M));
      GB_TRY(mega_start.alloc(M));
      k_mega_keys<<<grid_for(M, 256), 256, 0, s>>>(g->in.off.p, g->in.tgt.p, old_of.p, p->new_id.p, hot_of_blk.p,
                                                   p->nrows.p, B, mega_off.p, n_mega, M, deal, keys_in.p, vals_in.p);
      uint32_t row_bits = 1;
      while ((1u << row_bits) < n_mega) ++row_bits;
      size_t tb = 0;
      GB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, keys_in.p, mega_keys.p, vals_in.p, mega_vals.p, (int)M, 0,
                                              (int)(CB_MEGA_JBITS + row_bits), s));
      DevBuf<uint8_t> tmp;
      GB_TRY(tmp.alloc(tb));
      GB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, keys_in.p, mega_keys.p, vals_in.p, mega_vals.p, (int)M, 0,
                                              (int)(CB_MEGA_JBITS + row_bits), s));
      k_mega_starts<<<grid_for(M, 256), 256, 0, s>>>(mega_keys.p, M, mega_start.p);
      size_t sb = 0;
      GB_CUDA(cub::DeviceScan::InclusiveScan(nullptr, sb, mega_start.p, mega_start.p, cub::Max(), (int)M, s));
      DevBuf<uint8_t> stmp;
      GB_TRY(stmp.alloc(sb));
      GB_CUDA(cub::DeviceScan::InclusiveScan(stmp.p, sb, mega_start.p, mega_start.p, cub::Max(), (int)M, s));
      GB_CUDA(cudaMemsetAsync(lens.p, 0, (size_t)n_mega * 4, s));
      k_mega_counts<<<grid_for(M, 256), 256, 0, s>>>(mega_keys.p, mega_start.p, M, p->poff.p, goff.p, lens.p,
                                                     counters.p + 2);
      GB_CUDA(cudaGetLastError());
      GB_CUDA(cudaStreamSynchronize(s));  // keys_in / vals_in / tmp / stmp are released here
    }
    if (p->n_loc > p->n_cb)
      k_lens_tail<<<grid_for(p->n_loc - p->n_cb, 256), 256, 0, s>>>(indeg.p, p->n_cb, p->n_loc, deal, lens.p);
    if (p->S) {
      k_cb_groups<<<grid_for(p->S, 256), 256, 0, s>>>(goff.p, p->S);
      GB_TRY(scan_exclusive(s, goff.p, p->S + 1));
      uint32_t ng = 0;
      GB_CUDA(cudaMemcpyAsync(&ng, goff.p + p->S, 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      p->NG = ng;
    }
    {
      unsigned long long h[3] = {0, 0, 0};
      GB_CUDA(cudaMemcpyAsync(h, counters.p, 24, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      p->loc_edges = h[1];
      p->cb_edges = h[2];
    }
    // 5. SELL-32 layout of all local rows
    p->num_slices = (p->n_loc + 31) / 32;
    if (p->num_slices) {
      DevBuf<uint32_t> units, bases;
      GB_TRY(units.alloc(p->num_slices));
      GB_TRY(bases.alloc(p->num_slices));
      k_sell_widths<<<grid_for((uint64_t)p->num_slices * 32, 256), 256, 0, s>>>(lens.p, p->n_loc, p->num_slices, units.p);
      GB_CUDA(cudaMemcpyAsync(bases.p, units.p, (size_t)p->num_slices * 4, cudaMemcpyDeviceToDevice, s));
      GB_TRY(scan_exclusive(s, bases.p, p->num_slices));
      uint32_t last_base = 0, last_units = 0;
      GB_CUDA(cudaMemcpyAsync(&last_base, bases.p + p->num_slices - 1, 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaMemcpyAsync(&last_units, units.p + p->num_slices - 1, 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      const size_t total_units = (size_t)last_base + last_units;
      GB_TRY(p->slice_meta.alloc(p->num_slices));
      GB_TRY(p->sell.alloc(total_units, 64));
      GB_CUDA(cudaMemsetAsync(p->sell.p, 0xFF, (total_units + 64) * sizeof(uint4), s));  // ~0 = padding
      k_sell_meta<<<grid_for(p->num_slices, 256), 256, 0, s>>>(units.p, bases.p, p->num_slices, p->slice_meta.p);
      GB_CUDA(cudaGetLastError());
      GB_CUDA(cudaStreamSynchronize(s));
    }
    // 6. fill: segments + SELL remainders of the rows below n_cb, whole rows above
    GB_TRY(p->cb_ids.alloc(std::max<uint64_t>(p->NG, 1), 64));
    GB_TRY(p->cb_bits.alloc(p->NG / 32 + 4));
    GB_CUDA(cudaMemsetAsync(p->cb_bits.p, 0, (p->NG / 32 + 4) * 4, s));
    if (p->NG) {
      k_fill_u2<<<grid_for(p->NG + 64, 256), 256, 0, s>>>(p->cb_ids.p, p->NG + 64, make_uint2(B | (B << 16), B | (B << 16)));
      k_cb_bits<<<grid_for(p->S, 256), 256, 0, s>>>(goff.p, p->S, p->cb_bits.p);
      if (M)
        k_mega_fill<<<grid_for(M, 256), 256, 0, s>>>(mega_keys.p, mega_vals.p, mega_start.p, M, p->poff.p, p->blk.p, B,
                                                     goff.p, reinterpret_cast<uint16_t*>(p->cb_ids.p), p->slice_meta.p,
                                                     reinterpret_cast<uint32_t*>(p->sell.p));
      if (p->n_cb > n_mega)
        k_cb_fill<<<grid_for((uint64_t)(p->n_cb - n_mega) * 32, 256), 256, 0, s>>>(
            g->in.off.p, old_of.p, rec.p, p->poff.p, n_mega, p->n_cb, deal, goff.p,
            reinterpret_cast<uint16_t*>(p->cb_ids.p), p->slice_meta.p, reinterpret_cast<uint32_t*>(p->sell.p));
      GB_CUDA(cudaGetLastError());
      GB_CUDA(cudaStreamSynchronize(s));
    }
    if (p->n_loc > p->n_cb) {
      k_sell_fill_tail<<<grid_for((uint64_t)(p->num_slices - p->n_cb / 32) * 32, 256), 256, 0, s>>>(
          g->in.off.p, g->in.tgt.p, old_of.p, p->new_id.p, p->n_cb, p->n_loc, deal, p->num_slices, p->slice_meta.p,
          p->sell.p);
      GB_CUDA(cudaGetLastError());
    }
    // 7. chunks of the column-block kernel and every persistent CTA's share of them
    p->grid_cb = 0;
    p->trace = env_u32("GB_PR_TRACE", 0) != 0;
    if (p->NG) {
      // first group of every block's stream
      DevBuf<uint32_t> gbeg;
      GB_TRY(gbeg.alloc(p->KB + 1));
      k_gather_u32<<<grid_for(p->KB + 1, 128), 128, 0, s>>>(goff.p, p->poff.p, p->KB + 1, gbeg.p);
      std::vector<uint32_t> h_gbeg(p->KB + 1);
      GB_CUDA(cudaMemcpyAsync(h_gbeg.data(), gbeg.p, (size_t)(p->KB + 1) * 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      // ~8 tasks per SM keep the dynamic schedule level; a task is 32 chunks (one per warp) of 512..2048
      // groups (fewer, longer chunks = fewer segments cut by chunk boundaries); a thin block is cut into
      // >= 64 chunks (down to one 64-group step each) so that all warps share it — a lone warp runs at
      // its dependency latency, ~10x below the SM's throughput
      uint32_t C = env_u32("GB_PR_CHUNK", 0);
      const uint32_t T = CB_TASK_CHUNKS;
      if (!C) C = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(p->NG / ((uint64_t)dev_sms * 8 * T), 16384 / T), 65536 / T);
      C = std::max<uint32_t>(32u, (C + 31) / 32 * 32);
      p->chunk_groups = C;
      std::vector<uint32_t> h_cfirst(p->KB + 1, 0), h_cgrp(p->KB, C);
      std::vector<uint2> h_tasks;
      for (uint32_t j = 0; j < p->KB; ++j) {
        const uint32_t G = h_gbeg[j + 1] - h_gbeg[j];
        h_cgrp[j] = std::min<uint32_t>(C, std::max<uint32_t>(std::min<uint32_t>(64u, C), (G / 64 + 63) / 64 * 64));
        const uint32_t nc = (G + h_cgrp[j] - 1) / h_cgrp[j];
        h_cfirst[j + 1] = h_cfirst[j] + nc;
        for (uint32_t c = 0; c < nc; c += T)
          h_tasks.push_back(make_uint2(h_cfirst[j] + c, (std::min(nc, c + T) - c) | (j << 8)));
      }
      p->n_chunks = h_cfirst[p->KB];
      p->n_tasks = (uint32_t)h_tasks.size();
      p->grid_cb = (unsigned)std::min<uint64_t>(p->n_tasks, (uint64_t)dev_sms);  // one persistent CTA per SM
      GB_TRY(upload(s, &p->tasks, h_tasks));
      DevBuf<uint32_t> cfirst, cgrp;
      GB_TRY(upload(s, &cfirst, h_cfirst));
      GB_TRY(upload(s, &cgrp, h_cgrp));
      GB_TRY(p->chunks.alloc(p->n_chunks, 1));
      GB_TRY(p->tail_slot.alloc(p->n_chunks));
      GB_TRY(p->fix_list.alloc(p->n_chunks));
      GB_TRY(p->side.alloc((size_t)2 * p->n_chunks + 2));
      GB_CUDA(cudaMemsetAsync(p->side.p, 0, ((size_t)2 * p->n_chunks + 2) * 8, s));
      GB_CUDA(cudaMemsetAsync(p->chunks.p + p->n_chunks, 0, sizeof(uint4), s));  // sentinel: ends every fixup walk
      uint32_t* d_nfix = reinterpret_cast<uint32_t*>(counters.p + 3);
      k_cb_chunks<<<grid_for(p->n_chunks, 128), 128, 0, s>>>(goff.p, p->poff.p, p->nrows.p, gbeg.p, cfirst.p, cgrp.p,
                                                           p->KB, p->n_chunks, p->chunks.p, p->tail_slot.p,
                                                           p->fix_list.p, d_nfix);
      GB_CUDA(cudaGetLastError());
      uint32_t h_fix[2] = {0, 0};
      GB_CUDA(cudaMemcpyAsync(h_fix, d_nfix, 8, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      p->n_fix = h_fix[0];
      p->fix_max_row = h_fix[1];
    } else {
      GB_TRY(p->chunks.alloc(1));
      GB_TRY(p->tail_slot.alloc(1));
      GB_TRY(p->fix_list.alloc(1));
      GB_TRY(p->side.alloc(2));
      GB_TRY(p->tasks.alloc(1));
    }
    GB_TRY(p->task_ctr.alloc(std::max<unsigned>(p->grid_cb, 1)));
    GB_CUDA(cudaMemsetAsync(p->task_ctr.p, 0, (size_t)std::max<unsigned>(p->grid_cb, 1) * 4, s));
    GB_TRY(p->partial.alloc(std::max<uint64_t>(p->S, 1)));
    GB_CUDA(cudaMemsetAsync(p->partial.p, 0, std::max<uint64_t>(p->S, 1) * 4, s));
    GB_TRY(p->rem.alloc(std::max<uint32_t>(p->n_cb, 1)));
    {
      std::vector<uint32_t> h_kb((p->n_cb + 31) / 32);
      for (size_t w = 0; w < h_kb.size(); ++w) h_kb[w] = fin_blocks_of(h_nrows.data(), p->KB, (uint32_t)w * 32);
      GB_TRY(upload(s, &p->fin_kb, h_kb));
    }
    // 8. launch shapes and error buffers
    p->smem_cb = ((size_t)B + 4) * sizeof(float);
    GB_CUDA(cudaFuncSetAttribute(k_pr_cb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_cb));
    const uint64_t want_sell = ((uint64_t)p->num_slices + PR_SELL_THREADS / 32 - 1) / (PR_SELL_THREADS / 32);
    p->grid_sell = (unsigned)std::min<uint64_t>(want_sell, (uint64_t)dev_sms * 2);
    // rows with segments in more than SELL_FEW blocks are a prefix (nrows[] is non-increasing): k_pr_finish
    // completes them; all others are completed by their k_pr_sell lane (k_pr_cb is done by then)
    p->n_fin = p->KB > SELL_FEW ? std::min<uint32_t>(p->n_cb, (h_nrows[SELL_FEW] + 31) / 32 * 32) : 0;
    for (uint32_t j = 0; j < SELL_FEW && j < p->KB; ++j) {
      p->few_nrows[j] = h_nrows[j];
      p->few_poff[j] = h_poff[j];
    }
    p->n_fin_warp = p->KB > FIN_CTA_BLOCKS ? std::min<uint32_t>(p->n_fin, (h_nrows[FIN_CTA_BLOCKS] + 31) / 32 * 32) : 0;
    const uint64_t fin_warps2 = (uint64_t)p->n_fin_warp / 32 * (PR_FIN_THREADS / 32) + (p->n_fin - p->n_fin_warp + 63) / 64;
    const uint64_t fin_warps4 = (uint64_t)p->n_fin_warp / 32 * (PR_FIN_THREADS / 32) + (p->n_fin - p->n_fin_warp + 127) / 128;
    p->fin_u = (fin_warps2 + PR_FIN_THREADS / 32 - 1) / (PR_FIN_THREADS / 32) <= (uint64_t)dev_sms * 8 ? 2 : 4;
    const uint64_t fin_tasks = p->fin_u == 2 ? fin_warps2 : fin_warps4;
    const uint64_t want_fin = (fin_tasks + PR_FIN_THREADS / 32 - 1) / (PR_FIN_THREADS / 32);
    p->grid_fin = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(want_fin, (uint64_t)dev_sms * 8));
    // Role split of the finish CTAs: when every CTA has at most one pass of each kind to do (the grid is not
    // capped) and the hub chain is long (hundreds of blocks per row), CTAs [0, hub groups) take one hub
    // group each and the others the remaining rows — the two latency chains then run side by side instead
    // of one after the other in every CTA.  Measured (profiles/r02_sweep_breakdown.txt): -20 % on an
    // eighth-shard of RMAT-26; no gain when the grid is capped (RMAT-26 on one GPU) or the hub chain is
    // short (RMAT-22), where every CTA keeps doing both parts.
    p->fin_hub_ctas = 0;
    if (want_fin <= (uint64_t)dev_sms * 8 && p->KB > 4 * FIN_CTA_BLOCKS && p->n_fin_warp && p->n_fin > p->n_fin_warp &&
        p->grid_fin > p->n_fin_warp / 32)
      p->fin_hub_ctas = p->n_fin_warp / 32;
    const size_t nerr = (size_t)p->grid_sell + p->grid_fin;
    GB_TRY(p->block_err.alloc(nerr));
    GB_CUDA(cudaMemsetAsync(p->block_err.p, 0, nerr * sizeof(double), s));
    GB_TRY(p->err_hist.alloc(64));
    GB_TRY(p->ctrl.alloc(2));
    GB_CUDA(cudaMemsetAsync(p->ctrl.p, 0, 8, s));
    GB_CUDA(cudaStreamSynchronize(s));
    return GB_OK;
  }();
  if (st != GB_OK) {
    free_pr_plan(p);
    return st;
  }
  *out_plan = p;
  return GB_OK;
}

// The parts of segments cut by chunk boundaries are added by the first warps of k_pr_sell when every such
// row is completed later, by k_pr_finish (rows below n_fin).  A row that its k_pr_sell lane completes itself
// (few hot blocks: small graphs) needs the sum BEFORE that kernel: k_pr_fixup runs in between.
static bool fix_in_sell(const PrPlan* p) {
  return p->n_fix && p->grid_sell && p->fix_max_row < p->n_fin;
}
static PrArgs make_args(const PrPlan* p, float base, float damping, double tolerance) {
  PrArgs a{};
  a.outdeg = p->outdeg.p;
  a.n = p->n;
  a.deal = p->deal;
  a.n_loc = p->n_loc;
  a.n_cb = p->n_cb;
  a.n_fin_warp = p->n_fin_warp;
  a.fin_hub_ctas = p->fin_hub_ctas;
  a.n_fin = p->n_fin;
  a.few_kb = std::min<uint32_t>(p->KB, SELL_FEW);
  for (uint32_t j = 0; j < SELL_FEW; ++j) {
    a.few_nrows[j] = p->few_nrows[j];
    a.few_poff[j] = p->few_poff[j];
  }
  a.fix_in_sell = fix_in_sell(p) ? 1u : 0u;
  a.B = p->B;
  a.KB = p->KB;
  a.blk = p->blk.p;
  a.nrows = p->nrows.p;
  a.poff = p->poff.p;
  a.cb_ids = p->cb_ids.p;
  a.cb_bits = p->cb_bits.p;
  a.partial = p->partial.p;
  a.chunks = p->chunks.p;
  a.n_chunks = p->n_chunks;
  a.tail_slot = p->tail_slot.p;
  a.side = p->side.p;
  a.fix_list = p->fix_list.p;
  a.n_fix = p->n_fix;
  a.tasks = p->tasks.p;
  a.n_tasks = p->n_tasks;
  a.task_ctr = p->task_ctr.p;
  a.n_task_ranges = p->grid_cb;
  a.rem = p->rem.p;
  a.fin_kb = p->fin_kb.p;
  a.sell = p->sell.p;
  a.slice_meta = p->slice_meta.p;
  a.num_slices = p->num_slices;
  a.block_err = p->block_err.p;
  a.err_hist = p->err_hist.p;
  a.ctrl = p->ctrl.p;
  a.err_base_fin = p->grid_sell;
  a.base = base;
  a.damping = damping;
  a.tolerance = tolerance;
  a.n_peers = 0;
  a.mc_next = nullptr;
  return a;
}

// one sweep = column blocks (+ fixup of cut segments), SELL rows, then finish; *launches is advanced by
// the kernels launched
template <bool PEERS>
static gb_status launch_sweep(const PrPlan* p, const PrArgs& a, cudaStream_t s, uint64_t* launches) {
  cudaEvent_t* ev = nullptr;
  if (p->trace && p->trace_events.size() < 5 * 256) {
    const size_t base = p->trace_events.size();
    p->trace_events.resize(base + 5);
    for (int k = 0; k < 5; ++k) GB_CUDA(cudaEventCreate(&p->trace_events[base + k]));
    ev = &p->trace_events[base];
    GB_CUDA(cudaEventRecord(ev[0], s));
  }
  if (p->grid_cb) {
    k_pr_cb<<<p->grid_cb, PR_THREADS, p->smem_cb, s>>>(a);
    *launches += 1;
  }
  if (ev) GB_CUDA(cudaEventRecord(ev[1], s));
  if (p->n_fix && !a.fix_in_sell) {  // n_fix > 0 implies column blocks, so k_pr_cb ran
    k_pr_fixup<<<grid_for((uint64_t)p->n_fix * 32, 128, 296), 128, 0, s>>>(a);
    *launches += 1;
  }
  if (ev) GB_CUDA(cudaEventRecord(ev[2], s));
  if (p->grid_sell) {
    k_pr_sell<PEERS><<<p->grid_sell, PR_SELL_THREADS, 0, s>>>(a);
    *launches += 1;
  }
  if (ev) GB_CUDA(cudaEventRecord(ev[3], s));
  if (p->fin_u == 2) k_pr_finish<PEERS, 2><<<p->grid_fin, PR_FIN_THREADS, 0, s>>>(a);
  else k_pr_finish<PEERS, 4><<<p->grid_fin, PR_FIN_THREADS, 0, s>>>(a);
  if (ev) GB_CUDA(cudaEventRecord(ev[4], s));
  *launches += 1;
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

// ---- drivers ---------------------------------------------------------------------------------
static gb_status run_exact(const gb_graph* g, const gb_page_rank_config* cfg, float* d_scores,
                           uint64_t* ran, double* error) {
  cudaStream_t s = g->stream;
  DevBuf<float> out;
  DevBuf<uint64_t> d_ran;
  DevBuf<double> d_err;
  GB_TRY(out.alloc(g->n));
  GB_TRY(d_ran.alloc(1));
  GB_TRY(d_err.alloc(1));
  k_pr_exact<<<1, 32, 0, s>>>(g->in.off.p, g->in.tgt.p, g->out.off.p, g->n, cfg->max_iterations,
                             cfg->tolerance, cfg->damping_factor, d_scores, out.p, d_ran.p, d_err.p);
  GB_CUDA(cudaGetLastError());
  g->timing.kernel_launches += 1;
  GB_CUDA(cudaMemcpyAsync(ran, d_ran.p, 8, cudaMemcpyDeviceToHost, s));
  GB_CUDA(cudaMemcpyAsync(error, d_err.p, 8, cudaMemcpyDeviceToHost, s));
  GB_CUDA(cudaStreamSynchronize(s));
  return GB_OK;
}

static gb_status run_jacobi(const gb_graph* g, const gb_page_rank_config* cfg, float* d_scores,
                            uint64_t* ran, double* error) {
  if (!g->pr_plan) GB_TRY(build_pr_plan(g, PrDeal{}, &g->pr_plan));
  PrPlan* p = g->pr_plan;
  cudaStream_t s = g->stream;
  const uint32_t n = p->n;
  const float nf = (float)n;
  const float init = 1.0f / nf;                             // page_rank.rs:70
  const float base = (1.0f - cfg->damping_factor) / nf;     // page_rank.rs:71
  const bool profile = profiling_on();
  if (!p->x[0].p) {
    GB_TRY(p->x[0].alloc(n));
    GB_TRY(p->x[1].alloc(n));
    GB_TRY(p->scores.alloc(n));
  }

  k_pr_init<<<grid_for(n, 256), 256, 0, s>>>(n, p->n_active, init, base, p->deal, p->outdeg.p, p->x[0].p, p->x[1].p,
                                            p->scores.p);
  GB_CUDA(cudaMemsetAsync(p->ctrl.p, 0, 8, s));
  GB_CUDA(cudaMemsetAsync(p->task_ctr.p, 0, (size_t)std::max<unsigned>(p->grid_cb, 1) * 4, s));
  g->timing.kernel_launches += 1;

  PrArgs a = make_args(p, base, cfg->damping_factor, cfg->tolerance);
  a.scores = p->scores.p;

  // max_iterations == 0 never satisfies `iteration == max_iterations` (page_rank.rs:107): the
  // reference then runs until the tolerance is met; we bound that at 100000 sweeps.
  const uint64_t limit = cfg->max_iterations ? cfg->max_iterations : 100000ull;
  const bool can_stop_early = cfg->tolerance > 0.0;
  const uint32_t batch_cap = 64;
  uint64_t done = 0;      // sweeps launched so far
  uint64_t stopped = 0;   // sweep number at which the tolerance was met (0 = not yet)
  double last_err = 0.0;
  size_t ev_used = 0;
  while (done < limit && !stopped) {
    const uint32_t batch = (uint32_t)std::min<uint64_t>(limit - done, can_stop_early ? 8 : batch_cap);
    for (uint32_t b = 0; b < batch; ++b) {
      const uint64_t sweep_no = done + b + 1;
      a.x_cur = p->x[(sweep_no - 1) & 1].p;
      a.x_next = p->x[sweep_no & 1].p;
      a.sweep = b;
      a.sweep_no = (uint32_t)std::min<uint64_t>(sweep_no, 0xFFFFFFFFull);
      a.extra_err = (sweep_no == 1)
                        ? (double)(n - p->n_active) * fabs((double)(base - init))
                        : 0.0;
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      if (profile && ev_used + 2 <= 2 * PR_MAX_PROFILE_EVENTS) {
        while (p->prof_events.size() < ev_used + 2) {
          cudaEvent_t e;
          GB_CUDA(cudaEventCreate(&e));
          p->prof_events.push_back(e);
        }
        e0 = p->prof_events[ev_used];
        e1 = p->prof_events[ev_used + 1];
        ev_used += 2;
        GB_CUDA(cudaEventRecord(e0, s));
      }
      GB_TRY(launch_sweep<false>(p, a, s, &g->timing.kernel_launches));
      if (e1) GB_CUDA(cudaEventRecord(e1, s));
      if (sweep_no == 1 && p->n_active < n) {
        // sources without in-edges change exactly once (init/deg -> base/deg): patch the buffer
        // sweep 1 has just finished reading
        k_pr_fill_inactive<<<grid_for(n - p->n_active, 256), 256, 0, s>>>(n, p->n_active, base, p->outdeg.p,
                                                                         p->x[0].p);
        g->timing.kernel_launches += 1;
      }
    }
    GB_CUDA(cudaGetLastError());
    done += batch;
    if (can_stop_early || done >= limit) {
      uint32_t ctrl0 = 0;
      GB_CUDA(cudaMemcpyAsync(&ctrl0, p->ctrl.p, 4, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
      if (ctrl0 != 0) stopped = ctrl0;
      const uint64_t last = stopped ? stopped : done;
      const uint32_t slot = (uint32_t)(last - (done - batch) - 1);
      GB_CUDA(cudaMemcpyAsync(&last_err, p->err_hist.p + slot, 8, cudaMemcpyDeviceToHost, s));
      GB_CUDA(cudaStreamSynchronize(s));
    }
  }
  *ran = stopped ? stopped : done;
  *error = last_err;
  k_unpermute<<<grid_for(n, 256), 256, 0, s>>>(p->scores.p, p->new_id.p, n, d_scores);
  g->timing.kernel_launches += 1;
  GB_CUDA(cudaGetLastError());
  GB_CUDA(cudaStreamSynchronize(s));
  if (profile) {
    double ms = 0.0;
    for (size_t i = 0; i + 1 < ev_used; i += 2) {
      float t = 0.0f;
      GB_CUDA(cudaEventElapsedTime(&t, p->prof_events[i], p->prof_events[i + 1]));
      ms += t;
    }
    g->timing.hot_kernel_ms = ms;
    g->timing.hot_kernel_launches = ev_used / 2;
  }
  return GB_OK;
}

static gb_status page_rank_impl(const gb_graph* g, const gb_page_rank_config* cfg, float* d_scores,
                                float* h_scores, uint64_t* ran, double* error) {
  GB_REQUIRE(g && cfg && ran && error, "NULL argument");
  if (g->kind != GB_KIND_DIRECTED)
    return fail(GB_ERR_UNSUPPORTED, "page_rank needs a directed graph (page_rank.rs:61)");
  GB_REQUIRE(cfg->mode <= GB_PR_JACOBI, "bad page rank mode %u", cfg->mode);
  GB_REQUIRE(!(cfg->max_iterations == 0 && !(cfg->tolerance > 0.0)),
             "max_iterations == 0 with tolerance <= 0 never terminates (page_rank.rs:107)");
  DeviceGuard guard(g->device);
  std::lock_guard<std::mutex> lock(g->mu);
  cudaStream_t s = g->stream;
  uint32_t mode = cfg->mode;
  if (mode == GB_PR_AUTO) mode = (g->n <= 16384) ? GB_PR_EXACT : GB_PR_JACOBI;
  DevBuf<float> tmp_scores;
  if (!d_scores) {
    GB_TRY(tmp_scores.alloc(g->n));
    d_scores = tmp_scores.p;
  }
  if (mode == GB_PR_JACOBI && !g->pr_plan) GB_TRY(build_pr_plan(g, PrDeal{}, &g->pr_plan));  // not timed
  g->timing = gb_timing{};
  GB_CUDA(cudaEventRecord(g->ev_begin, s));
  if (mode == GB_PR_EXACT) GB_TRY(run_exact(g, cfg, d_scores, ran, error));
  else GB_TRY(run_jacobi(g, cfg, d_scores, ran, error));
  GB_CUDA(cudaEventRecord(g->ev_end, s));
  if (h_scores) GB_CUDA(cudaMemcpyAsync(h_scores, d_scores, (size_t)g->n * 4, cudaMemcpyDeviceToHost, s));
  GB_CUDA(cudaStreamSynchronize(s));
  float ms = 0.0f;
  GB_CUDA(cudaEventElapsedTime(&ms, g->ev_begin, g->ev_end));
  g->timing.total_ms = ms;
  return GB_OK;
}

}  // namespace gb

// ---- multi-GPU shard (1-D edge-cut by destination, 32-row slices dealt round-robin) ----------------
struct gb_pr_shard {
  const gb_graph* graph = nullptr;
  gb::PrPlan* plan = nullptr;
  gb::DevBuf<void*> sync_table;       // device copy of the ranks' control-block pointers (gb_pr_shard_sync)
  void* sync_table_host[8] = {nullptr};
};

extern "C" {

gb_status gb_pr_shard_create(const gb_graph* g, uint32_t rank, uint32_t world, gb_pr_shard** shard) {
  GB_REQUIRE(g && shard, "NULL argument");
  if (g->kind != GB_KIND_DIRECTED) return gb::fail(GB_ERR_UNSUPPORTED, "page rank shards need a directed graph");
  GB_REQUIRE(world >= 1 && rank < world, "bad shard %u of %u", rank, world);
  gb::DeviceGuard guard(g->device);
  std::lock_guard<std::mutex> lock(g->mu);
  gb_pr_shard* sh = new (std::nothrow) gb_pr_shard();
  if (!sh) return gb::fail(GB_ERR_OOM, "host allocation failed");
  sh->graph = g;
  gb::PrDeal deal;
  deal.P = world;
  deal.p = rank;
  gb_status st = gb::build_pr_plan(g, deal, &sh->plan);
  if (st != GB_OK) {
    delete sh;
    return st;
  }
  *shard = sh;
  return GB_OK;
}

gb_status gb_pr_shard_free(gb_pr_shard* shard) {
  if (!shard) return GB_OK;
  gb::DeviceGuard guard(shard->graph->device);
  gb::free_pr_plan(shard->plan);
  delete shard;
  return GB_OK;
}

gb_status gb_pr_shard_init(const gb_pr_shard* shard, float damping, float* d_x0, float* d_x1,
                           float* d_scores, void* cuda_stream) {
  GB_REQUIRE(shard && d_x0 && d_x1 && d_scores, "NULL argument");
  const gb_graph* g = shard->graph;
  const gb::PrPlan* p = shard->plan;
  gb::DeviceGuard guard(g->device);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const float nf = (float)p->n;
  const float init = 1.0f / nf;
  const float base = (1.0f - damping) / nf;
  // every rank fills the whole initial vector itself (no exchange needed before sweep 1)
  gb::k_pr_init<<<gb::grid_for(p->n, 256), 256, 0, s>>>(p->n, p->n_active, init, base, p->deal, p->outdeg.p, d_x0,
                                                       d_x1, d_scores);
  GB_CUDA(cudaMemsetAsync(p->ctrl.p, 0, 8, s));
  GB_CUDA(cudaMemsetAsync(p->task_ctr.p, 0, (size_t)std::max<unsigned>(p->grid_cb, 1) * 4, s));
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

gb_status gb_pr_shard_step(const gb_pr_shard* shard, float damping, uint64_t sweep_no, const float* d_x_cur,
                           float* d_x_next, float* const* d_peer_x_next, uint32_t peer_count,
                           float* d_mc_x_next, float* d_scores, double* d_error, void* cuda_stream) {
  GB_REQUIRE(shard && d_x_cur && d_x_next && d_scores && d_error, "NULL argument");
  GB_REQUIRE(peer_count <= 7, "at most 7 peers");
  GB_REQUIRE(peer_count == 0 || d_peer_x_next || d_mc_x_next, "peer pointer array is NULL");
  GB_REQUIRE(sweep_no >= 1, "sweep_no is 1-based");
  const gb_graph* g = shard->graph;
  const gb::PrPlan* p = shard->plan;
  gb::DeviceGuard guard(g->device);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const float nf = (float)p->n;
  const float init = 1.0f / nf;
  const float base = (1.0f - damping) / nf;
  gb::PrArgs a = gb::make_args(p, base, damping, -1.0 /* the caller owns the stop rule */);
  a.x_cur = d_x_cur;
  a.x_next = d_x_next;
  a.scores = d_scores;
  a.n_peers = d_mc_x_next ? 0 : peer_count;
  a.mc_next = d_mc_x_next;
  for (uint32_t i = 0; i < a.n_peers; ++i) a.peer_next[i] = d_peer_x_next[i];
  a.err_hist = d_error;
  a.sweep = 0;
  a.sweep_no = (uint32_t)std::min<uint64_t>(sweep_no, 0xFFFFFFFFull);
  // the closed-form error of the rows without in-edges is contributed once, by rank 0
  a.extra_err = (sweep_no == 1 && p->deal.p == 0)
                    ? (double)(p->n - p->n_active) * fabs((double)(base - init))
                    : 0.0;
  uint64_t launches = 0;
  if (peer_count || d_mc_x_next) GB_TRY(gb::launch_sweep<true>(p, a, s, &launches));
  else GB_TRY(gb::launch_sweep<false>(p, a, s, &launches));
  if (sweep_no == 1 && p->n_active < p->n)
    gb::k_pr_fill_inactive<<<gb::grid_for(p->n - p->n_active, 256), 256, 0, s>>>(
        p->n, p->n_active, base, p->outdeg.p, const_cast<float*>(d_x_cur));
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

gb_status gb_pr_shard_sync(const gb_pr_shard* shard, uint64_t sweep_no, const double* d_local_error,
                           void* d_self_block, void* const* d_peer_blocks, double* d_total_error,
                           uint32_t slot, void* cuda_stream) {
  GB_REQUIRE(shard && d_local_error && d_self_block && d_total_error, "NULL argument");
  const gb::PrPlan* p = shard->plan;
  GB_REQUIRE(p->deal.P <= 8, "at most 8 ranks");
  GB_REQUIRE(p->deal.P == 1 || d_peer_blocks, "peer block array is NULL");
  GB_REQUIRE(sweep_no >= 1 && sweep_no < 0x7FFFFFFFull, "bad sweep number");
  gb::DeviceGuard guard(shard->graph->device);
  cudaStream_t s = (cudaStream_t)cuda_stream;
  // the peer pointer table lives in the shard (device copy, refreshed when the pointers change)
  gb_pr_shard* sh = const_cast<gb_pr_shard*>(shard);
  void* table[8] = {nullptr};
  for (uint32_t q = 0; q < p->deal.P; ++q) table[q] = (q == p->deal.p) ? d_self_block : d_peer_blocks[q];
  if (!sh->sync_table.p || memcmp(table, sh->sync_table_host, sizeof table) != 0) {
    if (!sh->sync_table.p) GB_TRY(sh->sync_table.alloc(8));
    memcpy(sh->sync_table_host, table, sizeof table);
    GB_CUDA(cudaMemcpyAsync(sh->sync_table.p, table, sizeof table, cudaMemcpyHostToDevice, s));
  }
  gb::k_pr_sync<<<1, 32, 0, s>>>(static_cast<gb::PrSyncBlock*>(d_self_block),
                                reinterpret_cast<gb::PrSyncBlock* const*>(sh->sync_table.p), p->deal.P, p->deal.p,
                                (uint32_t)sweep_no, d_local_error, d_total_error, slot);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

gb_status gb_pr_shard_finish(const gb_pr_shard* shard, const float* d_scores_internal, float* d_scores_out,
                             void* cuda_stream) {
  GB_REQUIRE(shard && d_scores_internal && d_scores_out, "NULL argument");
  const gb_graph* g = shard->graph;
  const gb::PrPlan* p = shard->plan;
  gb::DeviceGuard guard(g->device);
  gb::k_unpermute<<<gb::grid_for(p->n, 256), 256, 0, (cudaStream_t)cuda_stream>>>(d_scores_internal, p->new_id.p,
                                                                                 p->n, d_scores_out);
  GB_CUDA(cudaGetLastError());
  return GB_OK;
}

gb_status gb_pr_shard_info(const gb_pr_shard* shard, gb_pr_shard_stats* stats) {
  GB_REQUIRE(shard && stats, "NULL argument");
  const gb::PrPlan* p = shard->plan;
  stats->rank = p->deal.p;
  stats->world = p->deal.P;
  stats->active_rows = p->n_active;
  stats->local_rows = p->n_loc;
  stats->local_edges = p->loc_edges;
  stats->block_edges = p->cb_edges;
  stats->block_entries = p->B;
  stats->hot_blocks = p->KB;
  stats->segments = p->S;
  stats->groups = p->NG;
  stats->chunks = p->n_chunks;
  stats->tasks = p->n_tasks;
  stats->cut_segments = p->n_fix;
  stats->chunk_groups = p->chunk_groups;
  stats->launches_per_sweep = 1 + (p->grid_cb ? 1 : 0) + (p->grid_sell ? 1 : 0) +
                              (p->grid_cb && p->n_fix && !gb::fix_in_sell(p) ? 1 : 0);
  stats->device_bytes = p->bytes();
  return GB_OK;
}

gb_status gb_page_rank_plan_info(const gb_graph* g, gb_pr_shard_stats* stats) {
  GB_REQUIRE(g && stats, "NULL argument");
  if (g->kind != GB_KIND_DIRECTED) return gb::fail(GB_ERR_UNSUPPORTED, "page rank needs a directed graph");
  gb::DeviceGuard guard(g->device);
  std::lock_guard<std::mutex> lock(g->mu);
  if (!g->pr_plan) GB_TRY(gb::build_pr_plan(g, gb::PrDeal{}, &g->pr_plan));
  gb_pr_shard tmp;
  tmp.graph = g;
  tmp.plan = g->pr_plan;
  return gb_pr_shard_info(&tmp, stats);
}

gb_status gb_page_rank_plan_reset(const gb_graph* g) {
  GB_REQUIRE(g, "NULL argument");
  gb::DeviceGuard guard(g->device);
  std::lock_guard<std::mutex> lock(g->mu);
  gb::free_pr_plan(g->pr_plan);
  g->pr_plan = nullptr;
  return GB_OK;
}

gb_status gb_page_rank(const gb_graph* graph, const gb_page_rank_config* config, float* scores,
                       uint64_t* ran_iterations, double* error) {
  GB_REQUIRE(scores != nullptr, "scores is NULL");
  return gb::page_rank_impl(graph, config, nullptr, scores, ran_iterations, error);
}

// One-shot PageRank of a host CSR.  The 4 bytes per edge of the targets dominate the upload, so they are
// streamed: offsets first, then the targets in row-aligned chunks on a copy stream, while the graph's own
// stream sorts the degrees, picks the hot blocks and classifies every chunk as it lands (TargetFeed in
// build_pr_plan).  Only the fill pass, the sweeps and the copy of the ranks run after the last byte.
// GB_PR_FEED_CHUNKS (default 16; 0 = upload everything, then build) and GB_PR_FEED_MIN_EDGES (default 2^22)
// are experiment knobs.
gb_status gb_page_rank_csr_u32(int device, uint32_t n, const uint32_t* in_off, const uint32_t* in_tgt,
                               const uint32_t* out_off, const gb_page_rank_config* config, float* scores,
                               uint64_t* ran_iterations, double* error) {
  GB_REQUIRE(scores != nullptr, "scores is NULL");
  GB_REQUIRE(n > 0, "node_count must be > 0");
  GB_REQUIRE(in_off && out_off, "offset arrays are NULL");
  GB_REQUIRE(in_off[n] == out_off[n], "in and out offsets disagree on the edge count");
  const uint64_t m = in_off[n];
  uint32_t chunks = gb::env_u32("GB_PR_FEED_CHUNKS", 16);
  if (m < gb::env_u32("GB_PR_FEED_MIN_EDGES", 1u << 22)) chunks = 0;
  // the single-warp EXACT mode (small graphs) reads the CSR directly: nothing to overlap
  if (!config || config->mode == GB_PR_EXACT || (config->mode == GB_PR_AUTO && n <= 16384)) chunks = 0;
  gb_graph* g = nullptr;
  GB_TRY(gb::new_graph(device, GB_KIND_DIRECTED, n, &g));
  if (chunks == 0) {
    gb_status st = gb::upload_host_csr(g->stream, n, in_off, in_tgt, nullptr, &g->in, "in");
    if (st == GB_OK) st = gb::upload_host_csr(g->stream, n, out_off, nullptr, nullptr, &g->out, "out");
    if (st == GB_OK) st = gb::page_rank_impl(g, config, nullptr, scores, ran_iterations, error);
    gb_graph_free(g);
    return st;
  }
  gb::TargetFeed feed;
  cudaStream_t copy = nullptr;
  cudaEvent_t offsets_in = nullptr;
  gb_status st = [&]() -> gb_status {
    GB_REQUIRE(in_off[0] == 0 && out_off[0] == 0, "offsets[0] must be 0");
    GB_REQUIRE(in_tgt != nullptr, "in targets is NULL");
    GB_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    GB_CUDA(cudaEventCreateWithFlags(&offsets_in, cudaEventDisableTiming));
    g->in.len = m;
    g->out.len = m;
    GB_TRY(g->in.off.alloc((size_t)n + 1));
    GB_TRY(g->out.off.alloc((size_t)n + 1));
    GB_TRY(g->in.tgt.alloc(m, 8));
    GB_CUDA(cudaMemcpyAsync(g->in.off.p, in_off, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, copy));
    GB_CUDA(cudaMemcpyAsync(g->out.off.p, out_off, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, copy));
    GB_CUDA(cudaEventRecord(offsets_in, copy));
    GB_CUDA(cudaMemsetAsync(g->in.tgt.p + m, 0, 8 * 4, copy));
    // chunk boundaries: rows, at about equal edge counts (a monotone in_off is checked on the device below;
    // a malformed one only makes uneven chunks here, the bounds stay inside [0, m])
    feed.row_begin.push_back(0);
    feed.edge_begin.push_back(0);
    for (uint32_t k = 1; k <= chunks; ++k) {
      uint32_t v = n;
      if (k < chunks) {
        const uint64_t want = m / chunks * k;
        v = (uint32_t)(std::upper_bound(in_off, in_off + n + 1, (uint32_t)want) - in_off);
        v = std::min(std::max(v, feed.row_begin.back()), n);
      }
      uint64_t e = std::min<uint64_t>(in_off[v], m);
      e = std::max(e, feed.edge_begin.back());
      if (k == chunks) e = m;
      feed.row_begin.push_back(v);
      feed.edge_begin.push_back(e);
    }
    for (uint32_t k = 0; k < chunks; ++k) {
      const uint64_t e0 = feed.edge_begin[k], e1 = feed.edge_begin[k + 1];
      if (e1 > e0)
        GB_CUDA(cudaMemcpyAsync(g->in.tgt.p + e0, in_tgt + e0, (e1 - e0) * 4, cudaMemcpyHostToDevice, copy));
      cudaEvent_t ev = nullptr;
      GB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      feed.ready.push_back(ev);
      GB_CUDA(cudaEventRecord(ev, copy));
    }
    // offsets: monotone, checked before anything indexes with them
    GB_CUDA(cudaStreamWaitEvent(g->stream, offsets_in, 0));
    gb::DevBuf<unsigned int> bad;
    GB_TRY(bad.alloc(2));
    GB_CUDA(cudaMemsetAsync(bad.p, 0, 8, g->stream));
    gb::k_feed_monotone<<<gb::grid_for(n, 256), 256, 0, g->stream>>>(g->in.off.p, n, bad.p);
    gb::k_feed_monotone<<<gb::grid_for(n, 256), 256, 0, g->stream>>>(g->out.off.p, n, bad.p + 1);
    unsigned int nbad[2] = {0, 0};
    GB_CUDA(cudaMemcpyAsync(nbad, bad.p, 8, cudaMemcpyDeviceToHost, g->stream));
    GB_CUDA(cudaStreamSynchronize(g->stream));
    {
      gb::DevBufStreamScope scope(g->stream);  // do not wait for the copy stream here
      bad.release();
    }
    GB_REQUIRE(nbad[0] == 0, "in offsets are not monotone (%u rows)", nbad[0]);
    GB_REQUIRE(nbad[1] == 0, "out offsets are not monotone (%u rows)", nbad[1]);
    g->feed = &feed;
    gb_status r = gb::page_rank_impl(g, config, nullptr, scores, ran_iterations, error);
    g->feed = nullptr;
    return r;
  }();
  g->feed = nullptr;
  if (copy) cudaStreamSynchronize(copy);  // an early error must not free buffers under a running copy
  gb_graph_free(g);
  for (cudaEvent_t ev : feed.ready) cudaEventDestroy(ev);
  if (offsets_in) cudaEventDestroy(offsets_in);
  if (copy) cudaStreamDestroy(copy);
  return st;
}

gb_status gb_digraph_for_page_rank_u32(int device, uint32_t n, const uint32_t* in_off, const uint32_t* in_tgt,
                                       const uint32_t* out_off, gb_graph** graph) {
  GB_REQUIRE(graph != nullptr, "graph is NULL");
  GB_REQUIRE(n > 0, "node_count must be > 0");
  GB_REQUIRE(in_off && out_off, "offset arrays are NULL");
  GB_REQUIRE(in_off[n] == out_off[n], "in and out offsets disagree on the edge count");
  gb_graph* g = nullptr;
  GB_TRY(gb::new_graph(device, GB_KIND_DIRECTED, n, &g));
  gb_status st = gb::upload_host_csr(g->stream, n, in_off, in_tgt, nullptr, &g->in, "in");
  if (st == GB_OK) st = gb::upload_host_csr(g->stream, n, out_off, nullptr, nullptr, &g->out, "out");
  if (st != GB_OK) {
    gb_graph_free(g);
    return st;
  }
  *graph = g;
  return GB_OK;
}

gb_status gb_page_rank_device(const gb_graph* graph, const gb_page_rank_config* config, float* d_scores,
                              uint64_t* ran_iterations, double* error) {
  GB_REQUIRE(d_scores != nullptr, "d_scores is NULL");
  return gb::page_rank_impl(graph, config, d_scores, nullptr, ran_iterations, error);
}

}  // extern "C"
