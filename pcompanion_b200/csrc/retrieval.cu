// Complementary retrieval: exact segment scoring + warp-level top-K, and top-K list merging.
//
// Replaces torch.matmul + torch.topk of /root/reference/src/models/p_companion.py:60-64 and
// /root/reference/src/utils/metrics.py:21,89, and the per-type filter -> matmul -> topk loop
// of /root/reference/inference.py:93-113.  Each score row ranks one contiguous run of catalog
// row ids (the members of its complementary type in a type-sorted permutation, or a plain
// slice of the catalog), which is exactly what the reference's per-type filter computes - the
// masked-out 99.9 % of a dense [R, P] score matrix is never formed.
//
// Scores are float64 sums of exact float32 x float32 products accumulated sequentially over
// d = 0 .. D-1 (one thread owns one (row, product) pair), mirrored by oracle/retrieval.py, so
// indices and scores match the oracle bit for bit; ties rank the lower catalog index first.
// Score rows that rank the same segment (same complementary type) are processed together, eight
// at a time, so a catalog row is fetched once per group instead of once per score row.
#include <math.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace pc {
namespace {

constexpr int TK_WARPS = 8;

struct Cand {
  double s;
  int64_t i;  // < 0: empty slot
};

// a ranks strictly before b
__device__ __forceinline__ bool ranks_before(double sa, int64_t ia, double sb, int64_t ib) {
  if (ib < 0) return ia >= 0;
  if (ia < 0) return false;
  return sa > sb || (sa == sb && ia < ib);
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ int64_t shfl_i64(int64_t v, int src) { return __shfl_sync(FULL, (long long)v, src); }

// Warp-distributed sorted list: lane j (< k) holds the j-th best entry.  Insert (s, i) - known to all lanes.
__device__ __forceinline__ void warp_topk_insert(Cand& mine, int k, double s, int64_t i) {
  const int lane = lane_id();
  const bool before = lane < k && ranks_before(s, i, mine.s, mine.i);
  const uint32_t mask = __ballot_sync(FULL, before);
  if (mask == 0) return;
  const int pos = __ffs(mask) - 1;
  const double up_s = __shfl_up_sync(FULL, mine.s, 1);
  const int64_t up_i = __shfl_up_sync(FULL, (long long)mine.i, 1);
  if (lane == pos) {
    mine.s = s;
    mine.i = i;
  } else if (lane > pos) {
    mine.s = up_s;
    mine.i = up_i;
  }
}

// Exclusion lists (pc_topk_by_type_excluding, pc_rank_remove_excluded): CSR lists of global product indices, ascending
// within each list (duplicates allowed).  Score row r uses list row_list[r] (list r when row_list is NULL); a list id
// outside [0, n_lists) means no exclusions.
struct Excl {
  const int64_t* offsets;
  const int64_t* idx;
  int64_t n_lists;
  const int32_t* row_list;
};

// [lo, hi) of score row `row`'s list
__device__ __forceinline__ void excl_bounds(const Excl ex, int64_t row, int64_t& lo, int64_t& hi) {
  const int64_t l = ex.row_list ? int64_t(ex.row_list[row]) : row;
  lo = hi = 0;
  if (l >= 0 && l < ex.n_lists) {
    lo = ex.offsets[l];
    hi = ex.offsets[l + 1];
  }
}

// g is among idx[lo .. hi) (ascending): binary search for the last entry <= g, on a pointer and a 32-bit count so that
// it fits the k <= 32 kernel's registers (a list holds < 2^31 entries)
__device__ __forceinline__ bool excl_listed(const int64_t* __restrict__ idx, int64_t lo, int64_t hi, int64_t g) {
  if (lo >= hi) return false;
  const int64_t* base = idx + lo;
  int n = int(hi - lo);
  while (n > 1) {
    const int half = n >> 1;
    if (base[half] <= g) base += half;
    n -= half;
  }
  return *base == g;
}

constexpr int RB = 8;            // score rows per group
constexpr int DCH = 16;          // dims per staged chunk
constexpr int TILE_LD = 20;      // floats per staged product chunk (16 + 4 pad: conflict-free LDS.128 across lanes)
constexpr int PP = 2;            // products per lane: every q value fetched from shared memory feeds PP fp64 chains.  With one
                                 // product per lane the kernel was bound by the shared-memory pipe (ncu: 0.73 LSU wavefronts
                                 // per SM cycle, fp64 pipe 24 % busy): 16 broadcast loads of q per 32 fp64 FMAs.
constexpr int BATCH = 32 * PP;   // products per warp per pass
constexpr int TILE_FLOATS = BATCH * TILE_LD;

// [sb, se): split `split` of `splits` of the run [beg, end), in pieces of a multiple of 32 positions
__device__ __forceinline__ void split_range(int64_t beg, int64_t end, int splits, int split, int64_t& sb, int64_t& se) {
  const int64_t len = end > beg ? end - beg : 0;
  const int64_t per = (ceil_div(len, int64_t(splits)) + 31) / 32 * 32;
  sb = beg + per * split;
  se = min(end, sb + per);
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = uint32_t(__cvta_generic_to_shared(smem_dst));
  const int bytes = valid ? 16 : 0;   // src-size 0 => the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(bytes) : "memory");
}

// stage the DCH-dim chunk `d0` of the warp's BATCH products (product p < 32: lane p's member[0], else lane p - 32's member[1]):
// 4 lanes cover the 64-byte piece of one product
__device__ __forceinline__ void stage_chunk(float* tile, const float* __restrict__ catalog, int dim, int d0, const int (&member)[PP]) {
  const int lane = lane_id();
#pragma unroll
  for (int j = 0; j < BATCH / 8; ++j) {
    const int prod = j * 8 + (lane >> 2);
    const int m = __shfl_sync(FULL, member[prod >> 5], prod & 31);
    const float* src = catalog + (m >= 0 ? int64_t(m) * dim + d0 + (lane & 3) * 4 : 0);
    cp_async16(tile + prod * TILE_LD + (lane & 3) * 4, src, m >= 0);
  }
}

// One pass of the scoring loop of topk_group_body (same staging, same arithmetic in the same order, so the same
// bits), for R query rows: acc[pp][r] = score of the lane's product cur[pp] against row r of q_s.  Chunk 0 of `cur`
// must already be in flight into tile[buf]; when `prefetch`, chunk 0 of `nxt` is put in flight during the last chunk.
// topk_group_body keeps its own inlined copy: folding it onto this helper reschedules the k <= 32 kernel's code.
template <int R>
__device__ __forceinline__ void score_pass(double (&acc)[PP][R], float* tile, int& buf, const double* q_s, int dim,
                                           const float* __restrict__ catalog, const int (&cur)[PP], const int (&nxt)[PP],
                                           bool prefetch) {
  const int lane = lane_id();
  const int n_chunks = dim / DCH;
#pragma unroll
  for (int pp = 0; pp < PP; ++pp)
#pragma unroll
    for (int r = 0; r < R; ++r) acc[pp][r] = 0.0;
  for (int c = 0; c < n_chunks; ++c) {
    if (c + 1 < n_chunks) stage_chunk(tile + (buf ^ 1) * TILE_FLOATS, catalog, dim, (c + 1) * DCH, cur);
    else if (prefetch) stage_chunk(tile + (buf ^ 1) * TILE_FLOATS, catalog, dim, 0, nxt);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncwarp();
    const float* mine_c = tile + buf * TILE_FLOATS + lane * TILE_LD;
    const double* qq = q_s + c * DCH;
#pragma unroll
    for (int j = 0; j < DCH / 4; ++j) {            // four dims at a time: PP x 4 converted values live in registers
      double cd[PP][4];
#pragma unroll
      for (int pp = 0; pp < PP; ++pp) {
        const float4 v = *reinterpret_cast<const float4*>(mine_c + pp * 32 * TILE_LD + 4 * j);
        cd[pp][0] = double(v.x); cd[pp][1] = double(v.y); cd[pp][2] = double(v.z); cd[pp][3] = double(v.w);
      }
#pragma unroll
      for (int dd = 0; dd < 4; dd += 2) {
#pragma unroll
        for (int r = 0; r < R; ++r) {   // PP x R independent accumulation chains, each sequential in d
          const double2 q2 = *reinterpret_cast<const double2*>(qq + r * dim + 4 * j + dd);
#pragma unroll
          for (int pp = 0; pp < PP; ++pp) {
            acc[pp][r] = fma(q2.x, cd[pp][dd], acc[pp][r]);
            acc[pp][r] = fma(q2.y, cd[pp][dd + 1], acc[pp][r]);
          }
        }
      }
    }
    __syncwarp();
    buf ^= 1;
  }
}

// grid = (splits, n_groups).  Group g = score rows row_ids[grp_begin[g] .. grp_begin[g+1]) (<= RB), all ranking
// members[seg_begin[g] .. seg_end[g]).  A lane owns PP products of a BATCH-product pass; 32-dim chunks are staged
// through shared memory with cp.async (double-buffered, coalesced), then every lane advances PP x RB independent
// sequential fp64 dot products (the chains interleave, which is what keeps the fp64 pipe busy).
// EXCL: a product whose global index is in its row's exclusion list never enters the row's list.  It is tested only
// after it ranks before the warp's current k-th entry, so the list is searched for few products.  The rows' list
// bounds sit in shared memory after the tile area (the k <= 32 kernel is capped at 128 registers).
template <bool EXCL>
__device__ __forceinline__ void topk_group_body(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                                                const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                                                int r_beg, int n_rows, int64_t beg, int64_t end, int k, int splits, int split,
                                                int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i,
                                                const Excl ex) {
  extern __shared__ double smem_d[];
  double* q_s = smem_d;                                                      // [RB][dim], rows >= n_rows are zero
  float* tiles = reinterpret_cast<float*>(q_s + RB * dim);                   // [TK_WARPS][2][BATCH][TILE_LD]
  Cand* lists = reinterpret_cast<Cand*>(tiles);                              // [TK_WARPS][RB][32], reuses the tile area after the scan
  int64_t* ex_lo = reinterpret_cast<int64_t*>(tiles + TK_WARPS * 2 * TILE_FLOATS);  // EXCL: [RB] list begin, then [RB] end
  static_assert(TK_WARPS * 2 * TILE_FLOATS * sizeof(float) >= TK_WARPS * RB * 32 * sizeof(Cand), "lists fit the tile area");
  const int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < RB * dim; i += blockDim.x) {
    const int r = i / dim, d = i - r * dim;
    q_s[i] = r < n_rows ? double(Q[int64_t(row_ids[r_beg + r]) * dim + d]) : 0.0;
  }
  if constexpr (EXCL) {
    if (threadIdx.x < RB) {
      int64_t lo = 0, hi = 0;
      if (int(threadIdx.x) < n_rows) excl_bounds(ex, row_ids[r_beg + threadIdx.x], lo, hi);
      ex_lo[threadIdx.x] = lo;
      ex_lo[RB + threadIdx.x] = hi;
    }
  }
  __syncthreads();
  int64_t sb, se;
  split_range(beg, end, splits, split, sb, se);
  Cand mine[RB];
#pragma unroll
  for (int r = 0; r < RB; ++r) mine[r] = Cand{-INFINITY, -1};
  float* tile = tiles + w * 2 * TILE_FLOATS;
  const int n_chunks = dim / DCH;
  auto member_at = [&](int64_t pos) -> int { return pos < se ? (members ? members[pos] : int(pos)) : -1; };

  int64_t base = sb + int64_t(w) * BATCH;
  int cur[PP], nxt[PP];
#pragma unroll
  for (int pp = 0; pp < PP; ++pp) cur[pp] = member_at(base + 32 * pp + lane);
  int buf = 0;
  if (base < se) stage_chunk(tile, catalog, dim, 0, cur);
  asm volatile("cp.async.commit_group;" ::: "memory");
  while (base < se) {
    const int64_t next_base = base + TK_WARPS * BATCH;
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) nxt[pp] = member_at(next_base + 32 * pp + lane);
    double acc[PP][RB];
#pragma unroll
    for (int pp = 0; pp < PP; ++pp)
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[pp][r] = 0.0;
    for (int c = 0; c < n_chunks; ++c) {
      if (c + 1 < n_chunks) stage_chunk(tile + (buf ^ 1) * TILE_FLOATS, catalog, dim, (c + 1) * DCH, cur);
      else if (next_base < se) stage_chunk(tile + (buf ^ 1) * TILE_FLOATS, catalog, dim, 0, nxt);
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      __syncwarp();
      const float* mine_c = tile + buf * TILE_FLOATS + lane * TILE_LD;
      const double* qq = q_s + c * DCH;
#pragma unroll
      for (int j = 0; j < DCH / 4; ++j) {            // four dims at a time: PP x 4 converted values live in registers
        double cd[PP][4];
#pragma unroll
        for (int pp = 0; pp < PP; ++pp) {
          const float4 v = *reinterpret_cast<const float4*>(mine_c + pp * 32 * TILE_LD + 4 * j);
          cd[pp][0] = double(v.x); cd[pp][1] = double(v.y); cd[pp][2] = double(v.z); cd[pp][3] = double(v.w);
        }
#pragma unroll
        for (int dd = 0; dd < 4; dd += 2) {
#pragma unroll
          for (int r = 0; r < RB; ++r) {   // PP x RB independent accumulation chains, each sequential in d
            const double2 q2 = *reinterpret_cast<const double2*>(qq + r * dim + 4 * j + dd);
#pragma unroll
            for (int pp = 0; pp < PP; ++pp) {
              acc[pp][r] = fma(q2.x, cd[pp][dd], acc[pp][r]);
              acc[pp][r] = fma(q2.y, cd[pp][dd + 1], acc[pp][r]);
            }
          }
        }
      }
      __syncwarp();
      buf ^= 1;
    }
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) {
      const int64_t gidx = cur[pp] >= 0 ? int64_t(cur[pp]) + index_base : -1;
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        if (r < n_rows) {
          const double thr_s = shfl_d(mine[r].s, k - 1);
          const int64_t thr_i = shfl_i64(mine[r].i, k - 1);
          bool take = gidx >= 0 && ranks_before(acc[pp][r], gidx, thr_s, thr_i);
          if constexpr (EXCL) take = take && !excl_listed(ex.idx, ex_lo[r], ex_lo[RB + r], gidx);
          uint32_t cand = __ballot_sync(FULL, take);
          while (cand) {
            const int src = __ffs(cand) - 1;
            cand &= cand - 1;
            warp_topk_insert(mine[r], k, shfl_d(acc[pp][r], src), shfl_i64(gidx, src));
          }
        }
      }
    }
    base = next_base;
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) cur[pp] = nxt[pp];
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();                 // every warp is done with its tiles: the area becomes the candidate lists
#pragma unroll
  for (int r = 0; r < RB; ++r) lists[(w * RB + r) * 32 + lane] = mine[r];
  __syncthreads();
  // warp r merges the TK_WARPS lists of row r
  if (w < n_rows) {
    Cand best = lists[(0 * RB + w) * 32 + lane];
    for (int ww = 1; ww < TK_WARPS; ++ww) {
      for (int j = 0; j < k; ++j) {
        const Cand c = lists[(ww * RB + w) * 32 + j];
        if (c.i < 0) break;
        warp_topk_insert(best, k, c.s, c.i);
      }
    }
    if (lane < k) {
      const int64_t o = (int64_t(row_ids[r_beg + w]) * splits + split) * k + lane;
      part_s[o] = best.s;
      part_i[o] = best.i;
    }
  }
}

__global__ void __launch_bounds__(TK_WARPS * 32, 2)
topk_groups_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                   const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                   const int32_t* __restrict__ grp_begin, const int64_t* __restrict__ seg_begin,
                   const int64_t* __restrict__ seg_end, int k, int splits, int64_t index_base,
                   double* __restrict__ part_s, int64_t* __restrict__ part_i) {
  const int g = blockIdx.y;
  const int r_beg = grp_begin[g];
  topk_group_body<false>(Q, dim, catalog, members, row_ids, r_beg, grp_begin[g + 1] - r_beg, seg_begin[g], seg_end[g], k,
                         splits, int(blockIdx.x), index_base, part_s, part_i, Excl{});
}

// ---- device-side grouping (pc_topk_by_type): no host read-back anywhere between the query upload and the result.
// keys[r] = type(r) << 32 | r (type = n_types for rows without a valid type: an empty run); after a stable sort on the
// type bytes, rows of one type are adjacent and ascending.  plan: position p starts a group iff its rank inside
// its type's run is a multiple of G (RB for k <= 32, the large-k kernel's rows per pass otherwise); grp_rows[p] =
// rows in that group (0 elsewhere).  The ranking kernel is launched with one CTA row per POSITION; the CTAs that do
// not start a group return at once.
__global__ void type_keys_kernel(const int32_t* __restrict__ row_type, int64_t rows, int n_types, uint64_t* __restrict__ keys) {
  const int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  int t = row_type ? row_type[r] : 0;
  if (t < 0 || t >= n_types) t = n_types;
  keys[r] = (uint64_t(uint32_t(t)) << 32) | uint64_t(uint32_t(r));
}

template <int G>
__global__ void topk_plan_kernel(const uint64_t* __restrict__ keys, int64_t rows, int32_t* __restrict__ row_ids,
                                 int32_t* __restrict__ grp_rows) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= rows) return;
  const uint64_t key = keys[p];
  const uint64_t t = key >> 32;
  row_ids[p] = int32_t(uint32_t(key));
  int64_t lo = 0, hi = p;                       // first position whose type is t
  const uint64_t want = t << 32;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < want) lo = mid + 1; else hi = mid;
  }
  int n = 0;
  if (((p - lo) % G) == 0) {
    n = 1;
    while (n < G && p + n < rows && (keys[p + n] >> 32) == t) ++n;
  }
  grp_rows[p] = n;
}

// pc_topk_by_type's ranking kernel (k <= 32).  EXCL: with exclusion lists (pc_topk_by_type_excluding); the plain
// instance ignores `ex`, which comes last so that the other parameters keep their offsets.
template <bool EXCL>
__global__ void __launch_bounds__(TK_WARPS * 32, 2)
topk_planned_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                    const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                    const int32_t* __restrict__ grp_rows, const uint64_t* __restrict__ keys,
                    const int64_t* __restrict__ type_offsets, int n_types, int64_t p0, int k, int splits,
                    int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i, const Excl ex) {
  const int64_t p = p0 + blockIdx.y;
  const int n_rows = grp_rows[p];
  if (n_rows == 0) return;                      // uniform over the CTA
  const int64_t t = int64_t(keys[p] >> 32);
  const int64_t beg = t < n_types ? type_offsets[t] : 0, end = t < n_types ? type_offsets[t + 1] : 0;
  topk_group_body<EXCL>(Q, dim, catalog, members, row_ids, int(p), n_rows, beg, end, k, splits, int(blockIdx.x), index_base,
                        part_s, part_i, ex);
}

// row-wise top-k of a materialised fp32 matrix: grid = (splits, rows)
__global__ void __launch_bounds__(TK_WARPS * 32)
topk_values_kernel(const float* __restrict__ V, int64_t cols, int k, int splits, double* __restrict__ part_s,
                   int64_t* __restrict__ part_i) {
  __shared__ Cand lists[TK_WARPS * 32];
  const int lane = lane_id(), w = warp_id();
  const int64_t r = blockIdx.y;
  const int split = blockIdx.x;
  const int64_t per = (ceil_div(cols, int64_t(splits)) + 31) / 32 * 32;
  const int64_t sb = per * split;
  const int64_t se = min(cols, sb + per);
  Cand mine{-INFINITY, -1};
  for (int64_t base = sb + int64_t(w) * 32; base < se; base += TK_WARPS * 32) {
    const int64_t c = base + lane;
    const bool valid = c < se;
    const double score = valid ? double(__ldg(V + r * cols + c)) : 0.0;
    const int64_t gidx = valid ? c : -1;
    const double thr_s = shfl_d(mine.s, k - 1);
    const int64_t thr_i = shfl_i64(mine.i, k - 1);
    uint32_t cand = __ballot_sync(FULL, valid && ranks_before(score, gidx, thr_s, thr_i));
    while (cand) {
      const int src = __ffs(cand) - 1;
      cand &= cand - 1;
      warp_topk_insert(mine, k, shfl_d(score, src), shfl_i64(gidx, src));
    }
  }
  lists[w * 32 + lane] = mine;
  __syncthreads();
  if (w == 0) {
    for (int ww = 1; ww < TK_WARPS; ++ww) {
      for (int j = 0; j < k; ++j) {
        const Cand c = lists[ww * 32 + j];
        if (c.i < 0) break;
        warp_topk_insert(mine, k, c.s, c.i);
      }
    }
    if (lane < k) {
      const int64_t o = (r * splits + split) * k + lane;
      part_s[o] = mine.s;
      part_i[o] = mine.i;
    }
  }
}

// one warp per row: merge `lists` sorted-or-not candidate lists of k entries
__global__ void __launch_bounds__(256)
topk_merge_kernel(const double* __restrict__ S, const int64_t* __restrict__ I, int64_t rows, int lists, int k,
                  double* __restrict__ out_s, int64_t* __restrict__ out_i) {
  const int64_t r = int64_t(blockIdx.x) * 8 + warp_id();
  if (r >= rows) return;
  const int lane = lane_id();
  Cand mine{-INFINITY, -1};
  const int64_t total = int64_t(lists) * k;
  for (int64_t base = 0; base < total; base += 32) {
    const int64_t c = base + lane;
    double s = -INFINITY;
    int64_t i = -1;
    if (c < total) {
      s = S[r * total + c];
      i = I[r * total + c];
    }
    uint32_t cand = __ballot_sync(FULL, i >= 0);
    while (cand) {
      const int src = __ffs(cand) - 1;
      cand &= cand - 1;
      warp_topk_insert(mine, k, shfl_d(s, src), shfl_i64(i, src));
    }
  }
  if (lane < k) {
    out_s[r * k + lane] = mine.s;
    out_i[r * k + lane] = mine.i;
  }
}

// ---- large k (WARP_K < k <= PC_TOPK_MAX_K).  The lists above hold one entry per lane.  For a larger k every (score
// row, CTA) keeps a candidate buffer in shared memory: [0, cnt) is the row's best entries at the last compaction
// (sorted, at most k) followed by the entries appended since.  An item is appended (warp-aggregated shared atomicAdd)
// when it ranks before the row's threshold, the k-th best entry at the last compaction (padding while fewer than k are
// held, so that everything enters).  When a buffer could overflow during the next pass, the CTA sorts every row's
// buffer (bitonic, ranking order) and keeps k.  All warps run the same number of passes so that they meet at the
// barriers.  (score, index) is a strict total order, so the selected entries do not depend on the append order.
constexpr int WARP_K = 32;                          // largest k of the warp-list kernels above
constexpr int LK_THREADS = TK_WARPS * 32;
constexpr int LK_GROUP_PASS = TK_WARPS * BATCH;     // items one pass of the group kernel can append to a row
constexpr int LK_STREAM_PASS = LK_THREADS;          // items one pass of the stream kernel can append

template <typename IdxT>
__device__ __forceinline__ void append_candidate(bool take, double s, IdxT i, double* bs, IdxT* bi, int* cnt) {
  const uint32_t mask = __ballot_sync(FULL, take);
  if (mask == 0) return;
  const int lane = lane_id(), leader = __ffs(mask) - 1;
  int slot = 0;
  if (lane == leader) slot = atomicAdd(cnt, __popc(mask));
  slot = __shfl_sync(FULL, slot, leader) + __popc(mask & ((1u << lane) - 1u));
  if (take) {
    bs[slot] = s;
    bi[slot] = i;
  }
}

// Sort the buffers of rows [0, n_rows) (row r at bs/bi + r * cap, cap a power of two), keep k, raise the thresholds.
// Called by the whole CTA after a barrier that follows the last append; ends with a barrier.
template <typename IdxT>
__device__ void compact_rows(double* bs, IdxT* bi, int cap, int* cnt, double* thr_s, IdxT* thr_i, int n_rows, int k) {
  int most = 0;
  for (int r = 0; r < n_rows; ++r) most = max(most, cnt[r]);
  int n2 = 2;                                       // sort length: a power of two >= every row's count, <= cap
  while (n2 < most) n2 <<= 1;
  const int ln2 = __ffs(n2) - 1;
  for (int t = threadIdx.x; t < n_rows * n2; t += blockDim.x) {
    const int r = t >> ln2, j = t & (n2 - 1);
    if (j >= cnt[r]) {
      bs[r * cap + j] = -INFINITY;
      bi[r * cap + j] = -1;
    }
  }
  __syncthreads();
  const int half = n2 >> 1;
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < n_rows * half; t += blockDim.x) {
        const int r = t >> (ln2 - 1), j = t & (half - 1);
        const int lo = ((j & ~(stride - 1)) << 1) | (j & (stride - 1)), hi = lo + stride;
        double* s = bs + r * cap;
        IdxT* i = bi + r * cap;
        const double sa = s[lo], sb = s[hi];
        const IdxT ia = i[lo], ib = i[hi];
        const bool best_first = (lo & size) == 0;   // direction of this run of the bitonic network
        if (best_first ? ranks_before(sb, ib, sa, ia) : ranks_before(sa, ia, sb, ib)) {
          s[lo] = sb; s[hi] = sa;
          i[lo] = ib; i[hi] = ia;
        }
      }
      __syncthreads();
    }
  }
  if (threadIdx.x < n_rows) {
    const int r = threadIdx.x, c = min(cnt[r], k);
    cnt[r] = c;
    thr_s[r] = c == k ? bs[r * cap + k - 1] : -INFINITY;
    thr_i[r] = c == k ? bi[r * cap + k - 1] : IdxT(-1);
  }
  __syncthreads();
}

// Large-k counterpart of topk_group_body for R score rows (R * cap buffer entries fit beside the staged tiles).  The
// scoring is score_pass, so the scores are the same bits as the k <= 32 kernel's.  EXCL: as topk_group_body, the
// exclusion test follows the threshold test; the list bounds follow `cnt` in shared memory.
template <int R, bool EXCL>
__device__ __forceinline__ void topk_group_large_body(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                                                      const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                                                      int r_beg, int n_rows, int64_t beg, int64_t end, int k, int cap, int splits,
                                                      int split, int64_t index_base, double* __restrict__ part_s,
                                                      int64_t* __restrict__ part_i, const Excl ex) {
  extern __shared__ double smem_d[];
  double* q_s = smem_d;                                                      // [R][dim], rows >= n_rows are zero
  float* tiles = reinterpret_cast<float*>(q_s + R * dim);                    // [TK_WARPS][2][BATCH][TILE_LD]
  double* bs = reinterpret_cast<double*>(tiles + TK_WARPS * 2 * TILE_FLOATS);  // [R][cap] scores
  double* thr_s = bs + R * cap;                                              // [R]
  int32_t* bi = reinterpret_cast<int32_t*>(thr_s + R);                       // [R][cap] catalog row ids
  int32_t* thr_i = bi + R * cap;                                             // [R]
  int* cnt = thr_i + R;                                                      // [R]
  int64_t* ex_lo = reinterpret_cast<int64_t*>((reinterpret_cast<uintptr_t>(cnt + R) + 7) & ~uintptr_t(7));  // EXCL: [R] begin, [R] end
  const int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < R * dim; i += blockDim.x) {
    const int r = i / dim, d = i - r * dim;
    q_s[i] = r < n_rows ? double(Q[int64_t(row_ids[r_beg + r]) * dim + d]) : 0.0;
  }
  if (threadIdx.x < R) {
    cnt[threadIdx.x] = 0;
    thr_s[threadIdx.x] = -INFINITY;
    thr_i[threadIdx.x] = -1;
    if constexpr (EXCL) {
      int64_t lo = 0, hi = 0;
      if (int(threadIdx.x) < n_rows) excl_bounds(ex, row_ids[r_beg + threadIdx.x], lo, hi);
      ex_lo[threadIdx.x] = lo;
      ex_lo[R + threadIdx.x] = hi;
    }
  }
  __syncthreads();
  int64_t sb, se;
  split_range(beg, end, splits, split, sb, se);
  const int64_t n_pass = se > sb ? ceil_div(se - sb, int64_t(LK_GROUP_PASS)) : 0;
  float* tile = tiles + w * 2 * TILE_FLOATS;
  auto member_at = [&](int64_t pos) -> int { return pos < se ? (members ? members[pos] : int(pos)) : -1; };

  int cur[PP], nxt[PP];
#pragma unroll
  for (int pp = 0; pp < PP; ++pp) cur[pp] = member_at(sb + int64_t(w) * BATCH + 32 * pp + lane);
  int buf = 0;
  if (n_pass > 0) stage_chunk(tile, catalog, dim, 0, cur);
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int64_t pass = 0; pass < n_pass; ++pass) {
    const int64_t next_base = sb + (pass + 1) * LK_GROUP_PASS + int64_t(w) * BATCH;
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) nxt[pp] = member_at(next_base + 32 * pp + lane);
    double acc[PP][R];
    score_pass<R>(acc, tile, buf, q_s, dim, catalog, cur, nxt, pass + 1 < n_pass);
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (r < n_rows) {
          bool take = cur[pp] >= 0 && ranks_before(acc[pp][r], cur[pp], thr_s[r], thr_i[r]);
          if constexpr (EXCL) take = take && !excl_listed(ex.idx, ex_lo[r], ex_lo[R + r], int64_t(cur[pp]) + index_base);
          append_candidate<int32_t>(take, acc[pp][r], cur[pp], bs + r * cap, bi + r * cap, cnt + r);
        }
      }
    }
    __syncthreads();                              // every append of this pass has landed
    bool full = false;
    for (int r = 0; r < n_rows; ++r) full |= cnt[r] > cap - LK_GROUP_PASS;
    __syncthreads();                              // every thread has read the counts before the next pass appends
    if (full) compact_rows<int32_t>(bs, bi, cap, cnt, thr_s, thr_i, n_rows, k);
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) cur[pp] = nxt[pp];
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  compact_rows<int32_t>(bs, bi, cap, cnt, thr_s, thr_i, n_rows, k);
  for (int t = threadIdx.x; t < n_rows * k; t += blockDim.x) {
    const int r = t / k, j = t - r * k;
    const int64_t o = (int64_t(row_ids[r_beg + r]) * splits + split) * k + j;
    const bool held = j < cnt[r];
    part_s[o] = held ? bs[r * cap + j] : -INFINITY;
    part_i[o] = held ? int64_t(bi[r * cap + j]) + index_base : -1;
  }
}

// grid = (splits, n_groups, RB / R): CTA z ranks rows [z * R, z * R + R) of its group (a group of <= RB rows is
// processed in sub-batches that each stream the segment)
template <int R>
__global__ void __launch_bounds__(LK_THREADS, 1)
topk_groups_large_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                         const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                         const int32_t* __restrict__ grp_begin, const int64_t* __restrict__ seg_begin,
                         const int64_t* __restrict__ seg_end, int k, int cap, int splits, int64_t index_base,
                         double* __restrict__ part_s, int64_t* __restrict__ part_i) {
  const int g = blockIdx.y;
  const int r_beg = grp_begin[g] + int(blockIdx.z) * R;
  const int n_rows = min(grp_begin[g + 1] - r_beg, R);
  if (n_rows <= 0) return;                      // uniform over the CTA
  topk_group_large_body<R, false>(Q, dim, catalog, members, row_ids, r_beg, n_rows, seg_begin[g], seg_end[g], k, cap,
                                  splits, int(blockIdx.x), index_base, part_s, part_i, Excl{});
}

// pc_topk_by_type's large-k ranking kernel: the plan formed groups of R rows, so one CTA ranks a whole group.  EXCL and
// `ex` as topk_planned_kernel.
template <int R, bool EXCL>
__global__ void __launch_bounds__(LK_THREADS, 1)
topk_planned_large_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                          const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                          const int32_t* __restrict__ grp_rows, const uint64_t* __restrict__ keys,
                          const int64_t* __restrict__ type_offsets, int n_types, int64_t p0, int k, int cap, int splits,
                          int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i, const Excl ex) {
  const int64_t p = p0 + blockIdx.y;
  const int n_rows = grp_rows[p];
  if (n_rows == 0) return;                      // uniform over the CTA
  const int64_t t = int64_t(keys[p] >> 32);
  const int64_t beg = t < n_types ? type_offsets[t] : 0, end = t < n_types ? type_offsets[t + 1] : 0;
  topk_group_large_body<R, EXCL>(Q, dim, catalog, members, row_ids, int(p), n_rows, beg, end, k, cap, splits,
                                 int(blockIdx.x), index_base, part_s, part_i, ex);
}

// Large-k selection over one row's stream of n (score, index) items, LK_STREAM_PASS items per pass; index < 0 is
// padding and never selected.  Writes k entries to out_s / out_i.  Shared memory: stream_smem_bytes(cap).
template <typename Load>
__device__ __forceinline__ void select_stream(int64_t n, int k, int cap, Load load, double* __restrict__ out_s,
                                              int64_t* __restrict__ out_i) {
  extern __shared__ double smem_d[];
  double* bs = smem_d;                                                       // [cap]
  double* thr_s = bs + cap;
  int64_t* bi = reinterpret_cast<int64_t*>(thr_s + 1);                       // [cap]
  int64_t* thr_i = bi + cap;
  int* cnt = reinterpret_cast<int*>(thr_i + 1);
  if (threadIdx.x == 0) {
    *cnt = 0;
    *thr_s = -INFINITY;
    *thr_i = -1;
  }
  __syncthreads();
  const int64_t n_pass = ceil_div(n, int64_t(LK_STREAM_PASS));
  for (int64_t pass = 0; pass < n_pass; ++pass) {
    const int64_t pos = pass * LK_STREAM_PASS + threadIdx.x;
    double s = -INFINITY;
    int64_t i = -1;
    if (pos < n) load(pos, s, i);
    append_candidate<int64_t>(i >= 0 && ranks_before(s, i, *thr_s, *thr_i), s, i, bs, bi, cnt);
    __syncthreads();                              // every append of this pass has landed
    const bool full = *cnt > cap - LK_STREAM_PASS;
    __syncthreads();                              // every thread has read the count before the next pass appends
    if (full) compact_rows<int64_t>(bs, bi, cap, cnt, thr_s, thr_i, 1, k);
  }
  compact_rows<int64_t>(bs, bi, cap, cnt, thr_s, thr_i, 1, k);
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    const bool held = j < *cnt;
    out_s[j] = held ? bs[j] : -INFINITY;
    out_i[j] = held ? bi[j] : -1;
  }
}

// large-k topk_values_kernel: grid = (splits, rows)
__global__ void __launch_bounds__(LK_THREADS)
topk_values_large_kernel(const float* __restrict__ V, int64_t cols, int k, int cap, int splits, double* __restrict__ part_s,
                         int64_t* __restrict__ part_i) {
  const int64_t r = blockIdx.y;
  const int split = blockIdx.x;
  const int64_t per = (ceil_div(cols, int64_t(splits)) + 31) / 32 * 32;
  const int64_t sb = per * split;
  const int64_t se = min(cols, sb + per);
  const float* row = V + r * cols + sb;
  const int64_t o = (r * splits + split) * k;
  select_stream(se > sb ? se - sb : 0, k, cap,
                [&](int64_t pos, double& s, int64_t& i) { s = double(__ldg(row + pos)); i = sb + pos; }, part_s + o, part_i + o);
}

// large-k topk_merge_kernel: one CTA per row
__global__ void __launch_bounds__(LK_THREADS)
topk_merge_large_kernel(const double* __restrict__ S, const int64_t* __restrict__ I, int lists, int k, int cap,
                        double* __restrict__ out_s, int64_t* __restrict__ out_i) {
  const int64_t r = blockIdx.x;
  const int64_t total = int64_t(lists) * k;
  select_stream(total, k, cap, [&](int64_t pos, double& s, int64_t& i) { s = S[r * total + pos]; i = I[r * total + pos]; },
                out_s + r * k, out_i + r * k);
}

// buffer capacity for k when a pass can append `pass` items: k kept entries, one pass and at least half a pass of
// slack (a power of two, for the bitonic sort)
int large_cap(int k, int pass) {
  int c = 1;
  while (c < k + pass + pass / 2) c <<= 1;
  return c;
}

constexpr size_t SMEM_BUDGET = 200 * 1024;   // most dynamic shared memory a group CTA may take (below the 227 KB per block)

// k <= 32 group kernels: the staged queries, then the tile area that the candidate lists reuse
size_t group_smem(int dim) {
  return size_t(RB) * dim * sizeof(double) +
         std::max(size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float), size_t(TK_WARPS) * RB * 32 * sizeof(Cand));
}

size_t group_large_smem(int rows, int cap, int dim) {
  return size_t(rows) * dim * sizeof(double) + size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float) +
         size_t(rows) * (cap + 1) * (sizeof(double) + sizeof(int32_t)) + size_t(rows) * sizeof(int);
}

// score rows one large-k group CTA ranks per pass over its segment: the most (a power of two <= RB) whose buffers fit
int group_large_rows(int cap, int dim) {
  int r = RB;
  while (r > 1 && group_large_smem(r, cap, dim) > SMEM_BUDGET) r >>= 1;
  return r;
}

// f(std::integral_constant<int, R>) for R = group_large_rows(cap, dim): the large-k group kernels are built for R = 8/4/2/1
template <typename F>
int with_large_rows(int cap, int dim, F f) {
  switch (group_large_rows(cap, dim)) {
    case 8: return f(std::integral_constant<int, 8>{});
    case 4: return f(std::integral_constant<int, 4>{});
    case 2: return f(std::integral_constant<int, 2>{});
    default: return f(std::integral_constant<int, 1>{});
  }
}

size_t stream_smem_bytes(int cap) { return size_t(cap + 1) * (sizeof(double) + sizeof(int64_t)) + sizeof(int); }

// gridDim.y is at most 65,535: launch(y0, ny) for every chunk [y0, y0 + ny) of the n rows or groups
template <typename Launch>
int launch_y_chunks(int64_t n, Launch launch) {
  for (int64_t y0 = 0; y0 < n; y0 += 65535) {
    launch(y0, unsigned(std::min<int64_t>(n - y0, 65535)));
    PC_LAUNCH_CHECK();
  }
  return PC_OK;
}

// With splits > 1, rank(ps, pi) writes every row's `splits` lists of k to split_ws ([rows][splits][k] scores, then the
// indices) and pc_topk_merge reduces them to the output; with one split it writes the output directly.
template <typename Rank>
int with_split_lists(int64_t rows, int k, int splits, void* split_ws, double* out_scores, int64_t* out_idx,
                     pc_stream_t stream, Rank rank) {
  double* ps = out_scores;
  int64_t* pi = out_idx;
  if (splits > 1) {
    ps = reinterpret_cast<double*>(split_ws);
    pi = reinterpret_cast<int64_t*>(ps + size_t(rows) * splits * k);
  }
  if (int rc = rank(ps, pi)) return rc;
  if (splits > 1) return pc_topk_merge(ps, pi, rows, splits, k, out_scores, out_idx, stream);
  return PC_OK;
}

// The device-side grouping of pc_topk_by_type(_excluding) and pc_rank_by_type in the first by_type_plan_bytes(rows) of
// the workspace: keys | sort workspace | row_ids | grp_rows.
size_t by_type_plan_bytes(int64_t rows) {
  if (rows <= 0) return 0;
  return align_up(size_t(rows) * 8, 256) + align_up(pc_sort_keys_workspace_bytes(rows), 256) + 2 * align_up(size_t(rows) * 4, 256);
}

struct ByTypePlan {
  const uint64_t* keys;
  const int32_t* row_ids;
  const int32_t* grp_rows;
};

// Sort the rows by type and mark groups of G rows (G: the rows per CTA of the ranking kernel that follows).
template <int G>
int plan_by_type(int64_t rows, int n_types, const int32_t* row_type, void* workspace, pc_stream_t stream, ByTypePlan& plan) {
  cudaStream_t st = as_stream(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  uint64_t* keys = reinterpret_cast<uint64_t*>(ws);             ws += align_up(size_t(rows) * 8, 256);
  void* sort_ws = ws;                                            const size_t sort_bytes = pc_sort_keys_workspace_bytes(rows);
  ws += align_up(sort_bytes, 256);
  int32_t* row_ids = reinterpret_cast<int32_t*>(ws);             ws += align_up(size_t(rows) * 4, 256);
  int32_t* grp_rows = reinterpret_cast<int32_t*>(ws);
  const unsigned tb = unsigned(ceil_div(rows, 256));
  type_keys_kernel<<<tb, 256, 0, st>>>(row_type, rows, n_types, keys);
  PC_LAUNCH_CHECK();
  // keys are created in ascending row order and the sort is stable: only the type bytes take part
  uint32_t mask = 0;
  for (int b = 0; b < 4; ++b)
    if ((uint64_t(n_types) >> (8 * b)) != 0) mask |= 1u << (4 + b);
  if (int rc = pc_sort_keys(keys, rows, mask, sort_ws, sort_bytes, stream)) return rc;
  topk_plan_kernel<G><<<tb, 256, 0, st>>>(keys, rows, row_ids, grp_rows);
  PC_LAUNCH_CHECK();
  plan = ByTypePlan{keys, row_ids, grp_rows};
  return PC_OK;
}

// ---- rank of a target (pc_rank_by_type).  The rank of row r's target is the number of products of the row's run that
// rank strictly before (s*, g) = (score of the target, its global index); it needs no selection state, only a count
// per row.  Counts are integers, so the CTAs of every split add into the zeroed out_rank in any order and the result is
// the same: no split lists and no merge.
__global__ void __launch_bounds__(TK_WARPS * 32, 2)
rank_planned_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                    const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                    const int32_t* __restrict__ grp_rows, const uint64_t* __restrict__ keys,
                    const int64_t* __restrict__ type_offsets, int n_types, int64_t p0, const float* __restrict__ target_rows,
                    const int64_t* __restrict__ target_idx, int splits, int64_t index_base,
                    unsigned long long* __restrict__ out_rank) {
  const int64_t p = p0 + blockIdx.y;
  const int n_rows = grp_rows[p];
  if (n_rows == 0) return;                      // uniform over the CTA
  const int64_t t = int64_t(keys[p] >> 32);
  if (t >= n_types) {                           // no valid type: the target can never be listed
    if (blockIdx.x == 0 && threadIdx.x < n_rows) out_rank[row_ids[p + threadIdx.x]] = ~0ull;
    return;
  }
  extern __shared__ double smem_d[];
  double* q_s = smem_d;                                                      // [RB][dim], rows >= n_rows are zero
  float* tiles = reinterpret_cast<float*>(q_s + RB * dim);                   // [TK_WARPS][2][BATCH][TILE_LD]
  double* tgt_s = reinterpret_cast<double*>(tiles + TK_WARPS * 2 * TILE_FLOATS);  // [RB] target scores
  int64_t* tgt_i = reinterpret_cast<int64_t*>(tgt_s + RB);                   // [RB] target global indices
  unsigned long long* cnt_s = reinterpret_cast<unsigned long long*>(tgt_i + RB);  // [RB] CTA counts
  const int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < RB * dim; i += blockDim.x) {
    const int r = i / dim, d = i - r * dim;
    q_s[i] = r < n_rows ? double(Q[int64_t(row_ids[p + r]) * dim + d]) : 0.0;
  }
  if (threadIdx.x < RB) cnt_s[threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x < RB) {
    // the arithmetic of score_pass in its order (sequential in d, fma(q, c, acc) from 0): the target's streamed score
    // has the same bits, so the target never ranks before itself
    const int r = threadIdx.x;
    double acc = 0.0;
    int64_t g = -1;
    if (r < n_rows) {
      const int64_t row = row_ids[p + r];
      const float* tr = target_rows + row * dim;
      for (int d = 0; d < dim; ++d) acc = fma(q_s[r * dim + d], double(tr[d]), acc);
      g = target_idx[row];
    }
    tgt_s[r] = acc;
    tgt_i[r] = g;
  }
  __syncthreads();
  int64_t sb, se;
  split_range(type_offsets[t], type_offsets[t + 1], splits, int(blockIdx.x), sb, se);
  float* tile = tiles + w * 2 * TILE_FLOATS;
  auto member_at = [&](int64_t pos) -> int { return pos < se ? (members ? members[pos] : int(pos)) : -1; };

  unsigned cnt[RB];
#pragma unroll
  for (int r = 0; r < RB; ++r) cnt[r] = 0;
  int64_t base = sb + int64_t(w) * BATCH;
  int cur[PP], nxt[PP];
#pragma unroll
  for (int pp = 0; pp < PP; ++pp) cur[pp] = member_at(base + 32 * pp + lane);
  int buf = 0;
  if (base < se) stage_chunk(tile, catalog, dim, 0, cur);
  asm volatile("cp.async.commit_group;" ::: "memory");
  while (base < se) {                           // warps advance independently: nothing shared is written in the loop
    const int64_t next_base = base + TK_WARPS * BATCH;
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) nxt[pp] = member_at(next_base + 32 * pp + lane);
    double acc[PP][RB];
    score_pass<RB>(acc, tile, buf, q_s, dim, catalog, cur, nxt, next_base < se);
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) {
      const int64_t gidx = int64_t(cur[pp]) + index_base;
#pragma unroll
      for (int r = 0; r < RB; ++r)
        cnt[r] += (cur[pp] >= 0 && ranks_before(acc[pp][r], gidx, tgt_s[r], tgt_i[r])) ? 1u : 0u;
    }
    base = next_base;
#pragma unroll
    for (int pp = 0; pp < PP; ++pp) cur[pp] = nxt[pp];
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const unsigned c = __reduce_add_sync(FULL, cnt[r]);
    if (lane == 0 && r < n_rows && c) atomicAdd(cnt_s + r, (unsigned long long)c);
  }
  __syncthreads();
  if (threadIdx.x < n_rows && cnt_s[threadIdx.x]) atomicAdd(out_rank + row_ids[p + threadIdx.x], cnt_s[threadIdx.x]);
}

// s = sum_d q[d] * c[d] with the streaming pass's arithmetic in its order: fma(double(q[d]), double(c[d]), s), d ascending
// from 0 (dim % 16 == 0, rows 16-byte aligned)
__device__ __forceinline__ double dot_stream_order(const float* __restrict__ q, const float* __restrict__ c, int dim) {
  double s = 0.0;
  for (int d = 0; d < dim; d += 4) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(q + d)), b = __ldg(reinterpret_cast<const float4*>(c + d));
    s = fma(double(a.x), double(b.x), s);
    s = fma(double(a.y), double(b.y), s);
    s = fma(double(a.z), double(b.z), s);
    s = fma(double(a.w), double(b.w), s);
  }
  return s;
}

// pc_rank_remove_excluded: one warp per score row, lanes stride the row's list.  An entry is subtracted when it is
// distinct (not equal to its predecessor), local, of the row's type and ranks strictly before the target.  Both scores
// have the streaming pass's bits, so every subtracted entry is one that pc_rank_by_type counted, and a target listed
// in its own list never is.
__global__ void __launch_bounds__(256, 4)
rank_remove_excluded_kernel(const float* __restrict__ Q, int64_t rows, int dim, const float* __restrict__ catalog,
                            int64_t n_products, const int32_t* __restrict__ type_id, const int32_t* __restrict__ row_type,
                            const float* __restrict__ target_rows, const int64_t* __restrict__ target_idx,
                            int64_t index_base, const Excl ex, int64_t* __restrict__ inout_rank) {
  const int64_t r = int64_t(blockIdx.x) * 8 + warp_id();
  if (r >= rows) return;                        // uniform over the warp, as every early return below
  const int64_t rank = inout_rank[r];
  if (rank < 0) return;
  int64_t lo, hi;
  excl_bounds(ex, r, lo, hi);
  if (lo >= hi) return;
  const int lane = lane_id();
  const float* qr = Q + r * dim;
  const double ts = dot_stream_order(qr, target_rows + r * dim, dim);
  const int64_t tg = target_idx[r];
  const int t = row_type ? row_type[r] : 0;
  unsigned c = 0;
  for (int64_t j = lo + lane; j < hi; j += 32) {
    const int64_t e = ex.idx[j];
    const int64_t loc = e - index_base;
    if ((j > lo && ex.idx[j - 1] == e) || loc < 0 || loc >= n_products) continue;
    if (row_type && type_id[loc] != t) continue;
    c += ranks_before(dot_stream_order(qr, catalog + loc * dim, dim), e, ts, tg) ? 1u : 0u;
  }
  c = __reduce_add_sync(FULL, c);
  if (lane == 0 && c) inout_rank[r] = rank - int64_t(c);
}

}  // namespace
}  // namespace pc

using namespace pc;

extern "C" size_t pc_topk_groups_workspace_bytes(int64_t rows, int k, int splits) {
  if (rows <= 0 || k <= 0 || splits <= 1) return 0;
  return size_t(rows) * size_t(splits) * size_t(k) * (sizeof(double) + sizeof(int64_t));
}

extern "C" int pc_topk_groups(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                              const int32_t* row_ids, const int32_t* grp_begin, const int64_t* seg_begin,
                              const int64_t* seg_end, int64_t n_groups, int k, int splits, int64_t index_base,
                              double* out_scores, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                              pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && n_groups >= 0, PC_ERR_INVALID, "topk_groups: negative size");
  if (rows == 0 || n_groups == 0) return PC_OK;
  PC_REQUIRE(q && catalog && row_ids && grp_begin && seg_begin && seg_end && out_scores && out_idx, PC_ERR_INVALID,
             "topk_groups: null pointer");
  PC_REQUIRE(k >= 1 && k <= PC_TOPK_MAX_K, PC_ERR_UNSUPPORTED, "topk_groups: k=%d outside [1,%d]", k, PC_TOPK_MAX_K);
  PC_REQUIRE(dim >= DCH && dim % DCH == 0 && dim <= 1024, PC_ERR_UNSUPPORTED, "topk_groups: dim=%d must be a multiple of %d (<= 1024)", dim, DCH);
  PC_REQUIRE(splits >= 1 && splits <= 65535, PC_ERR_UNSUPPORTED, "topk_groups: bad splits");
  PC_REQUIRE(splits == 1 || (workspace && workspace_bytes >= pc_topk_groups_workspace_bytes(rows, k, splits)),
             PC_ERR_WORKSPACE, "topk_groups: workspace too small");
  cudaStream_t st = as_stream(stream);
  return with_split_lists(rows, k, splits, workspace, out_scores, out_idx, stream, [&](double* ps, int64_t* pi) -> int {
    if (k > WARP_K) {
      const int cap = large_cap(k, LK_GROUP_PASS);
      return with_large_rows(cap, dim, [&](auto rows_per_cta) -> int {
        constexpr int R = decltype(rows_per_cta)::value;
        const size_t smem = group_large_smem(R, cap, dim);
        PC_CUDA(cudaFuncSetAttribute(topk_groups_large_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        return launch_y_chunks(n_groups, [&](int64_t g0, unsigned ng) {
          topk_groups_large_kernel<R><<<dim3(splits, ng, RB / R), LK_THREADS, smem, st>>>(
              q, dim, catalog, members, row_ids, grp_begin + g0, seg_begin + g0, seg_end + g0, k, cap, splits, index_base,
              ps, pi);
        });
      });
    }
    const size_t smem = group_smem(dim);
    PC_CUDA(cudaFuncSetAttribute(topk_groups_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SMEM_BUDGET)));
    PC_REQUIRE(smem <= SMEM_BUDGET, PC_ERR_UNSUPPORTED, "topk_groups: shared memory budget exceeded");
    return launch_y_chunks(n_groups, [&](int64_t g0, unsigned ng) {
      topk_groups_kernel<<<dim3(splits, ng, 1), TK_WARPS * 32, smem, st>>>(q, dim, catalog, members, row_ids, grp_begin + g0,
                                                                          seg_begin + g0, seg_end + g0, k, splits, index_base,
                                                                          ps, pi);
    });
  });
}

extern "C" size_t pc_topk_by_type_workspace_bytes(int64_t rows, int k, int splits) {
  return by_type_plan_bytes(rows) + pc_topk_groups_workspace_bytes(rows, k, splits);
}

// pc_topk_by_type (EXCL = false, `ex` ignored) and pc_topk_by_type_excluding: the same grouping, splits and merge
template <bool EXCL>
static int topk_by_type_impl(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                             const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                             int64_t index_base, double* out_scores, int64_t* out_idx, void* workspace,
                             size_t workspace_bytes, const Excl ex, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && rows < (int64_t(1) << 31), PC_ERR_INVALID, "topk_by_type: bad row count");
  if (rows == 0) return PC_OK;
  PC_REQUIRE(q && catalog && type_offsets && out_scores && out_idx && workspace, PC_ERR_INVALID, "topk_by_type: null pointer");
  PC_REQUIRE(n_types >= 1 && n_types < (1 << 30), PC_ERR_INVALID, "topk_by_type: bad n_types=%d", n_types);
  PC_REQUIRE(k >= 1 && k <= PC_TOPK_MAX_K, PC_ERR_UNSUPPORTED, "topk_by_type: k=%d outside [1,%d]", k, PC_TOPK_MAX_K);
  PC_REQUIRE(dim >= DCH && dim % DCH == 0 && dim <= 1024, PC_ERR_UNSUPPORTED, "topk_by_type: dim=%d must be a multiple of %d (<= 1024)", dim, DCH);
  PC_REQUIRE(splits >= 1 && splits <= 65535, PC_ERR_UNSUPPORTED, "topk_by_type: bad splits");
  PC_REQUIRE(workspace_bytes >= pc_topk_by_type_workspace_bytes(rows, k, splits), PC_ERR_WORKSPACE, "topk_by_type: workspace too small");
  cudaStream_t st = as_stream(stream);
  void* split_ws = reinterpret_cast<char*>(workspace) + by_type_plan_bytes(rows);
  return with_split_lists(rows, k, splits, split_ws, out_scores, out_idx, stream, [&](double* ps, int64_t* pi) -> int {
    ByTypePlan plan;
    if (k > WARP_K) {
      const int cap = large_cap(k, LK_GROUP_PASS);
      return with_large_rows(cap, dim, [&](auto rows_per_cta) -> int {
        constexpr int R = decltype(rows_per_cta)::value;
        if (int rc = plan_by_type<R>(rows, n_types, row_type, workspace, stream, plan)) return rc;
        const size_t smem = group_large_smem(R, cap, dim) + (EXCL ? 8 + 2 * R * sizeof(int64_t) : 0);   // + aligned list bounds
        PC_CUDA(cudaFuncSetAttribute(topk_planned_large_kernel<R, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        return launch_y_chunks(rows, [&](int64_t p0, unsigned np) {
          topk_planned_large_kernel<R, EXCL><<<dim3(splits, np, 1), LK_THREADS, smem, st>>>(
              q, dim, catalog, members, plan.row_ids, plan.grp_rows, plan.keys, type_offsets, n_types, p0, k, cap, splits,
              index_base, ps, pi, ex);
        });
      });
    }
    if (int rc = plan_by_type<RB>(rows, n_types, row_type, workspace, stream, plan)) return rc;
    const size_t smem = group_smem(dim);
    PC_REQUIRE(smem <= SMEM_BUDGET, PC_ERR_UNSUPPORTED, "topk_by_type: shared memory budget exceeded");
    PC_CUDA(cudaFuncSetAttribute(topk_planned_kernel<EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(SMEM_BUDGET)));
    const size_t smem_ex = smem + (EXCL ? 2 * RB * sizeof(int64_t) : 0);   // + the rows' list bounds after the tile area
    return launch_y_chunks(rows, [&](int64_t p0, unsigned np) {
      topk_planned_kernel<EXCL><<<dim3(splits, np, 1), TK_WARPS * 32, smem_ex, st>>>(
          q, dim, catalog, members, plan.row_ids, plan.grp_rows, plan.keys, type_offsets, n_types, p0, k, splits, index_base,
          ps, pi, ex);
    });
  });
}

extern "C" int pc_topk_by_type(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                               const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                               int64_t index_base, double* out_scores, int64_t* out_idx, void* workspace,
                               size_t workspace_bytes, pc_stream_t stream) {
  return topk_by_type_impl<false>(q, rows, dim, catalog, members, type_offsets, n_types, row_type, k, splits, index_base,
                                  out_scores, out_idx, workspace, workspace_bytes, Excl{}, stream);
}

extern "C" int pc_topk_by_type_excluding(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                                         const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                                         int64_t index_base, const int64_t* excl_offsets, const int64_t* excl_idx,
                                         int64_t n_lists, const int32_t* row_list, double* out_scores, int64_t* out_idx,
                                         void* workspace, size_t workspace_bytes, pc_stream_t stream) {
  PC_REQUIRE(n_lists >= 0, PC_ERR_INVALID, "topk_by_type_excluding: n_lists=%lld < 0", (long long)n_lists);
  PC_REQUIRE(n_lists == 0 || (excl_offsets && excl_idx), PC_ERR_INVALID, "topk_by_type_excluding: null exclusion lists");
  const Excl ex{excl_offsets, excl_idx, n_lists, row_list};
  return topk_by_type_impl<true>(q, rows, dim, catalog, members, type_offsets, n_types, row_type, k, splits, index_base,
                                 out_scores, out_idx, workspace, workspace_bytes, ex, stream);
}

extern "C" size_t pc_rank_by_type_workspace_bytes(int64_t rows) { return by_type_plan_bytes(rows); }

extern "C" int pc_rank_by_type(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                               const int64_t* type_offsets, int n_types, const int32_t* row_type, const float* target_rows,
                               const int64_t* target_idx, int splits, int64_t index_base, int64_t* out_rank, void* workspace,
                               size_t workspace_bytes, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && rows < (int64_t(1) << 31), PC_ERR_INVALID, "rank_by_type: bad row count");
  if (rows == 0) return PC_OK;
  PC_REQUIRE(q && catalog && type_offsets && target_rows && target_idx && out_rank && workspace, PC_ERR_INVALID,
             "rank_by_type: null pointer");
  PC_REQUIRE(n_types >= 1 && n_types < (1 << 30), PC_ERR_INVALID, "rank_by_type: bad n_types=%d", n_types);
  PC_REQUIRE(dim >= DCH && dim % DCH == 0 && dim <= 1024, PC_ERR_UNSUPPORTED, "rank_by_type: dim=%d must be a multiple of %d (<= 1024)", dim, DCH);
  PC_REQUIRE(splits >= 1 && splits <= 65535, PC_ERR_UNSUPPORTED, "rank_by_type: bad splits");
  PC_REQUIRE(workspace_bytes >= pc_rank_by_type_workspace_bytes(rows), PC_ERR_WORKSPACE, "rank_by_type: workspace too small");
  cudaStream_t st = as_stream(stream);
  PC_CUDA(cudaMemsetAsync(out_rank, 0, size_t(rows) * sizeof(int64_t), st));
  ByTypePlan plan;
  if (int rc = plan_by_type<RB>(rows, n_types, row_type, workspace, stream, plan)) return rc;
  const size_t smem = size_t(RB) * dim * sizeof(double) + size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float) +
                      size_t(RB) * (sizeof(double) + sizeof(int64_t) + sizeof(unsigned long long));
  PC_CUDA(cudaFuncSetAttribute(rank_planned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  return launch_y_chunks(rows, [&](int64_t p0, unsigned np) {
    rank_planned_kernel<<<dim3(splits, np, 1), TK_WARPS * 32, smem, st>>>(
        q, dim, catalog, members, plan.row_ids, plan.grp_rows, plan.keys, type_offsets, n_types, p0, target_rows, target_idx,
        splits, index_base, reinterpret_cast<unsigned long long*>(out_rank));
  });
}

extern "C" int pc_rank_remove_excluded(const float* q, int64_t rows, int dim, const float* catalog, int64_t n_products,
                                       const int32_t* type_id, const int32_t* row_type, const float* target_rows,
                                       const int64_t* target_idx, int64_t index_base, const int64_t* excl_offsets,
                                       const int64_t* excl_idx, int64_t n_lists, const int32_t* row_list,
                                       int64_t* inout_rank, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && n_products >= 0 && n_lists >= 0, PC_ERR_INVALID, "rank_remove_excluded: negative size");
  if (rows == 0 || n_lists == 0 || n_products == 0) return PC_OK;
  PC_REQUIRE(q && catalog && target_rows && target_idx && excl_offsets && excl_idx && inout_rank, PC_ERR_INVALID,
             "rank_remove_excluded: null pointer");
  PC_REQUIRE(!row_type || type_id, PC_ERR_INVALID, "rank_remove_excluded: row_type needs type_id");
  PC_REQUIRE(dim >= DCH && dim % DCH == 0 && dim <= 1024, PC_ERR_UNSUPPORTED, "rank_remove_excluded: dim=%d must be a multiple of %d (<= 1024)", dim, DCH);
  const Excl ex{excl_offsets, excl_idx, n_lists, row_list};
  rank_remove_excluded_kernel<<<unsigned(ceil_div(rows, 8)), 256, 0, as_stream(stream)>>>(
      q, rows, dim, catalog, n_products, type_id, row_type, target_rows, target_idx, index_base, ex, inout_rank);
  PC_LAUNCH_CHECK();
  return PC_OK;
}

extern "C" int pc_topk_merge(const double* scores, const int64_t* idx, int64_t rows, int lists, int k,
                             double* out_scores, int64_t* out_idx, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && lists >= 1, PC_ERR_INVALID, "topk_merge: bad sizes");
  if (rows == 0) return PC_OK;
  PC_REQUIRE(scores && idx && out_scores && out_idx, PC_ERR_INVALID, "topk_merge: null pointer");
  PC_REQUIRE(k >= 1 && k <= PC_TOPK_MAX_K, PC_ERR_UNSUPPORTED, "topk_merge: k=%d outside [1,%d]", k, PC_TOPK_MAX_K);
  if (k > WARP_K) {
    PC_REQUIRE(rows < (int64_t(1) << 31), PC_ERR_UNSUPPORTED, "topk_merge: rows=%lld too many for k > %d", (long long)rows, WARP_K);
    const int cap = large_cap(k, LK_STREAM_PASS);
    topk_merge_large_kernel<<<unsigned(rows), LK_THREADS, stream_smem_bytes(cap), as_stream(stream)>>>(
        scores, idx, lists, k, cap, out_scores, out_idx);
    PC_LAUNCH_CHECK();
    return PC_OK;
  }
  topk_merge_kernel<<<unsigned(ceil_div(rows, 8)), 256, 0, as_stream(stream)>>>(scores, idx, rows, lists, k,
                                                                                out_scores, out_idx);
  PC_LAUNCH_CHECK();
  return PC_OK;
}

extern "C" size_t pc_topk_rows_workspace_bytes(int64_t rows, int k, int splits) {
  return pc_topk_groups_workspace_bytes(rows, k, splits);
}

extern "C" int pc_topk_rows(const float* values, int64_t rows, int64_t cols, int k, int splits, double* out_scores,
                            int64_t* out_idx, void* workspace, size_t workspace_bytes, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && cols >= 0 && cols < (int64_t(1) << 31), PC_ERR_INVALID, "topk_rows: bad sizes");
  if (rows == 0) return PC_OK;
  PC_REQUIRE(values && out_scores && out_idx, PC_ERR_INVALID, "topk_rows: null pointer");
  PC_REQUIRE(k >= 1 && k <= PC_TOPK_MAX_K, PC_ERR_UNSUPPORTED, "topk_rows: k=%d outside [1,%d]", k, PC_TOPK_MAX_K);
  PC_REQUIRE(splits >= 1 && splits <= 65535, PC_ERR_UNSUPPORTED, "topk_rows: bad splits");
  PC_REQUIRE(splits == 1 || (workspace && workspace_bytes >= pc_topk_rows_workspace_bytes(rows, k, splits)),
             PC_ERR_WORKSPACE, "topk_rows: workspace too small");
  cudaStream_t st = as_stream(stream);
  return with_split_lists(rows, k, splits, workspace, out_scores, out_idx, stream, [&](double* ps, int64_t* pi) {
    return launch_y_chunks(rows, [&](int64_t r0, unsigned nr) {
      const dim3 grid{unsigned(splits), nr, 1u};
      if (k > WARP_K) {
        const int cap = large_cap(k, LK_STREAM_PASS);
        topk_values_large_kernel<<<grid, LK_THREADS, stream_smem_bytes(cap), st>>>(values + r0 * cols, cols, k, cap, splits,
                                                                                  ps + r0 * splits * k, pi + r0 * splits * k);
      } else {
        topk_values_kernel<<<grid, TK_WARPS * 32, 0, st>>>(values + r0 * cols, cols, k, splits, ps + r0 * splits * k,
                                                           pi + r0 * splits * k);
      }
    });
  });
}
