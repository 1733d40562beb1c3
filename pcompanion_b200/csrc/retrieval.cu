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

constexpr int RB = 8;            // score rows per group
constexpr int DCH = 16;          // dims per staged chunk
constexpr int TILE_LD = 20;      // floats per staged product chunk (16 + 4 pad: conflict-free LDS.128 across lanes)
constexpr int PP = 2;            // products per lane: every q value fetched from shared memory feeds PP fp64 chains.  With one
                                 // product per lane the kernel was bound by the shared-memory pipe (ncu: 0.73 LSU wavefronts
                                 // per SM cycle, fp64 pipe 24 % busy): 16 broadcast loads of q per 32 fp64 FMAs.
constexpr int BATCH = 32 * PP;   // products per warp per pass
constexpr int TILE_FLOATS = BATCH * TILE_LD;

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
__device__ __forceinline__ void topk_group_body(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                                                const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                                                int r_beg, int n_rows, int64_t beg, int64_t end, int k, int splits, int split,
                                                int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i) {
  extern __shared__ double smem_d[];
  double* q_s = smem_d;                                                      // [RB][dim], rows >= n_rows are zero
  float* tiles = reinterpret_cast<float*>(q_s + RB * dim);                   // [TK_WARPS][2][BATCH][TILE_LD]
  Cand* lists = reinterpret_cast<Cand*>(tiles);                              // [TK_WARPS][RB][32], reuses the tile area after the scan
  const int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < RB * dim; i += blockDim.x) {
    const int r = i / dim, d = i - r * dim;
    q_s[i] = r < n_rows ? double(Q[int64_t(row_ids[r_beg + r]) * dim + d]) : 0.0;
  }
  __syncthreads();
  const int64_t len = end > beg ? end - beg : 0;
  const int64_t per = (ceil_div(len, int64_t(splits)) + 31) / 32 * 32;
  const int64_t sb = beg + per * split;
  const int64_t se = min(end, sb + per);
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
          uint32_t cand = __ballot_sync(FULL, gidx >= 0 && ranks_before(acc[pp][r], gidx, thr_s, thr_i));
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
  topk_group_body(Q, dim, catalog, members, row_ids, r_beg, grp_begin[g + 1] - r_beg, seg_begin[g], seg_end[g], k, splits,
                  int(blockIdx.x), index_base, part_s, part_i);
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

__global__ void __launch_bounds__(TK_WARPS * 32, 2)
topk_planned_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                    const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                    const int32_t* __restrict__ grp_rows, const uint64_t* __restrict__ keys,
                    const int64_t* __restrict__ type_offsets, int n_types, int64_t p0, int k, int splits,
                    int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i) {
  const int64_t p = p0 + blockIdx.y;
  const int n_rows = grp_rows[p];
  if (n_rows == 0) return;                      // uniform over the CTA
  const int64_t t = int64_t(keys[p] >> 32);
  const int64_t beg = t < n_types ? type_offsets[t] : 0, end = t < n_types ? type_offsets[t + 1] : 0;
  topk_group_body(Q, dim, catalog, members, row_ids, int(p), n_rows, beg, end, k, splits, int(blockIdx.x), index_base,
                  part_s, part_i);
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
// scoring is score_pass, so the scores are the same bits as the k <= 32 kernel's.
template <int R>
__device__ __forceinline__ void topk_group_large_body(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                                                      const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                                                      int r_beg, int n_rows, int64_t beg, int64_t end, int k, int cap, int splits,
                                                      int split, int64_t index_base, double* __restrict__ part_s,
                                                      int64_t* __restrict__ part_i) {
  extern __shared__ double smem_d[];
  double* q_s = smem_d;                                                      // [R][dim], rows >= n_rows are zero
  float* tiles = reinterpret_cast<float*>(q_s + R * dim);                    // [TK_WARPS][2][BATCH][TILE_LD]
  double* bs = reinterpret_cast<double*>(tiles + TK_WARPS * 2 * TILE_FLOATS);  // [R][cap] scores
  double* thr_s = bs + R * cap;                                              // [R]
  int32_t* bi = reinterpret_cast<int32_t*>(thr_s + R);                       // [R][cap] catalog row ids
  int32_t* thr_i = bi + R * cap;                                             // [R]
  int* cnt = thr_i + R;                                                      // [R]
  const int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < R * dim; i += blockDim.x) {
    const int r = i / dim, d = i - r * dim;
    q_s[i] = r < n_rows ? double(Q[int64_t(row_ids[r_beg + r]) * dim + d]) : 0.0;
  }
  if (threadIdx.x < R) {
    cnt[threadIdx.x] = 0;
    thr_s[threadIdx.x] = -INFINITY;
    thr_i[threadIdx.x] = -1;
  }
  __syncthreads();
  const int64_t len = end > beg ? end - beg : 0;
  const int64_t per = (ceil_div(len, int64_t(splits)) + 31) / 32 * 32;
  const int64_t sb = beg + per * split;
  const int64_t se = min(end, sb + per);
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
          const bool take = cur[pp] >= 0 && ranks_before(acc[pp][r], cur[pp], thr_s[r], thr_i[r]);
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
  topk_group_large_body<R>(Q, dim, catalog, members, row_ids, r_beg, n_rows, seg_begin[g], seg_end[g], k, cap, splits,
                           int(blockIdx.x), index_base, part_s, part_i);
}

// pc_topk_by_type's large-k ranking kernel: the plan formed groups of R rows, so one CTA ranks a whole group
template <int R>
__global__ void __launch_bounds__(LK_THREADS, 1)
topk_planned_large_kernel(const float* __restrict__ Q, int dim, const float* __restrict__ catalog,
                          const int32_t* __restrict__ members, const int32_t* __restrict__ row_ids,
                          const int32_t* __restrict__ grp_rows, const uint64_t* __restrict__ keys,
                          const int64_t* __restrict__ type_offsets, int n_types, int64_t p0, int k, int cap, int splits,
                          int64_t index_base, double* __restrict__ part_s, int64_t* __restrict__ part_i) {
  const int64_t p = p0 + blockIdx.y;
  const int n_rows = grp_rows[p];
  if (n_rows == 0) return;                      // uniform over the CTA
  const int64_t t = int64_t(keys[p] >> 32);
  const int64_t beg = t < n_types ? type_offsets[t] : 0, end = t < n_types ? type_offsets[t + 1] : 0;
  topk_group_large_body<R>(Q, dim, catalog, members, row_ids, int(p), n_rows, beg, end, k, cap, splits, int(blockIdx.x),
                           index_base, part_s, part_i);
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

size_t group_large_smem(int rows, int cap, int dim) {
  return size_t(rows) * dim * sizeof(double) + size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float) +
         size_t(rows) * (cap + 1) * (sizeof(double) + sizeof(int32_t)) + size_t(rows) * sizeof(int);
}

// score rows one large-k group CTA ranks per pass over its segment: the most (a power of two <= RB) whose buffers fit
int group_large_rows(int cap, int dim) {
  int r = RB;
  while (r > 1 && group_large_smem(r, cap, dim) > 200 * 1024) r >>= 1;
  return r;
}

size_t stream_smem_bytes(int cap) { return size_t(cap + 1) * (sizeof(double) + sizeof(int64_t)) + sizeof(int); }

template <int R>
int launch_groups_large(const float* q, int dim, const float* catalog, const int32_t* members, const int32_t* row_ids,
                        const int32_t* grp_begin, const int64_t* seg_begin, const int64_t* seg_end, int64_t n_groups, int k,
                        int cap, int splits, int64_t index_base, double* ps, int64_t* pi, cudaStream_t st) {
  const size_t smem = group_large_smem(R, cap, dim);
  PC_CUDA(cudaFuncSetAttribute(topk_groups_large_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  for (int64_t g0 = 0; g0 < n_groups; g0 += 65535) {   // gridDim.y limit
    const int64_t ng = n_groups - g0 < 65535 ? n_groups - g0 : 65535;
    dim3 grid{unsigned(splits), unsigned(ng), unsigned(RB / R)};
    topk_groups_large_kernel<R><<<grid, LK_THREADS, smem, st>>>(q, dim, catalog, members, row_ids, grp_begin + g0,
                                                               seg_begin + g0, seg_end + g0, k, cap, splits, index_base, ps, pi);
    PC_LAUNCH_CHECK();
  }
  return PC_OK;
}

template <int R>
int launch_by_type_large(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                         const int64_t* type_offsets, int n_types, const uint64_t* keys, int32_t* row_ids, int32_t* grp_rows,
                         int k, int cap, int splits, int64_t index_base, double* ps, int64_t* pi, cudaStream_t st) {
  topk_plan_kernel<R><<<unsigned(ceil_div(rows, 256)), 256, 0, st>>>(keys, rows, row_ids, grp_rows);
  PC_LAUNCH_CHECK();
  const size_t smem = group_large_smem(R, cap, dim);
  PC_CUDA(cudaFuncSetAttribute(topk_planned_large_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  for (int64_t p0 = 0; p0 < rows; p0 += 65535) {   // gridDim.y limit
    const int64_t np = rows - p0 < 65535 ? rows - p0 : 65535;
    dim3 grid{unsigned(splits), unsigned(np), 1u};
    topk_planned_large_kernel<R><<<grid, LK_THREADS, smem, st>>>(q, dim, catalog, members, row_ids, grp_rows, keys,
                                                                type_offsets, n_types, p0, k, cap, splits, index_base, ps, pi);
    PC_LAUNCH_CHECK();
  }
  return PC_OK;
}

int groups_large(const float* q, int dim, const float* catalog, const int32_t* members, const int32_t* row_ids,
                 const int32_t* grp_begin, const int64_t* seg_begin, const int64_t* seg_end, int64_t n_groups, int k,
                 int splits, int64_t index_base, double* ps, int64_t* pi, cudaStream_t st) {
  const int cap = large_cap(k, LK_GROUP_PASS);
  switch (group_large_rows(cap, dim)) {
    case 8: return launch_groups_large<8>(q, dim, catalog, members, row_ids, grp_begin, seg_begin, seg_end, n_groups, k, cap, splits, index_base, ps, pi, st);
    case 4: return launch_groups_large<4>(q, dim, catalog, members, row_ids, grp_begin, seg_begin, seg_end, n_groups, k, cap, splits, index_base, ps, pi, st);
    case 2: return launch_groups_large<2>(q, dim, catalog, members, row_ids, grp_begin, seg_begin, seg_end, n_groups, k, cap, splits, index_base, ps, pi, st);
    default: return launch_groups_large<1>(q, dim, catalog, members, row_ids, grp_begin, seg_begin, seg_end, n_groups, k, cap, splits, index_base, ps, pi, st);
  }
}

int by_type_large(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                  const int64_t* type_offsets, int n_types, const uint64_t* keys, int32_t* row_ids, int32_t* grp_rows, int k,
                  int splits, int64_t index_base, double* ps, int64_t* pi, cudaStream_t st) {
  const int cap = large_cap(k, LK_GROUP_PASS);
  switch (group_large_rows(cap, dim)) {
    case 8: return launch_by_type_large<8>(q, rows, dim, catalog, members, type_offsets, n_types, keys, row_ids, grp_rows, k, cap, splits, index_base, ps, pi, st);
    case 4: return launch_by_type_large<4>(q, rows, dim, catalog, members, type_offsets, n_types, keys, row_ids, grp_rows, k, cap, splits, index_base, ps, pi, st);
    case 2: return launch_by_type_large<2>(q, rows, dim, catalog, members, type_offsets, n_types, keys, row_ids, grp_rows, k, cap, splits, index_base, ps, pi, st);
    default: return launch_by_type_large<1>(q, rows, dim, catalog, members, type_offsets, n_types, keys, row_ids, grp_rows, k, cap, splits, index_base, ps, pi, st);
  }
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
  cudaStream_t st = as_stream(stream);
  const size_t smem = size_t(RB) * dim * sizeof(double) +
                      std::max(size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float), size_t(TK_WARPS) * RB * 32 * sizeof(Cand));
  PC_CUDA(cudaFuncSetAttribute(topk_groups_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PC_REQUIRE(smem <= 200 * 1024, PC_ERR_UNSUPPORTED, "topk_groups: shared memory budget exceeded");
  double* ps = out_scores;
  int64_t* pi = out_idx;
  if (splits > 1) {
    PC_REQUIRE(workspace && workspace_bytes >= pc_topk_groups_workspace_bytes(rows, k, splits), PC_ERR_WORKSPACE,
               "topk_groups: workspace too small");
    ps = reinterpret_cast<double*>(workspace);
    pi = reinterpret_cast<int64_t*>(ps + size_t(rows) * splits * k);
  }
  if (k > WARP_K) {
    if (int rc = groups_large(q, dim, catalog, members, row_ids, grp_begin, seg_begin, seg_end, n_groups, k, splits,
                              index_base, ps, pi, st))
      return rc;
  } else {
    for (int64_t g0 = 0; g0 < n_groups; g0 += 65535) {   // gridDim.y limit
      const int64_t ng = n_groups - g0 < 65535 ? n_groups - g0 : 65535;
      dim3 grid{unsigned(splits), unsigned(ng), 1u};
      topk_groups_kernel<<<grid, TK_WARPS * 32, smem, st>>>(q, dim, catalog, members, row_ids, grp_begin + g0, seg_begin + g0,
                                                            seg_end + g0, k, splits, index_base, ps, pi);
      PC_LAUNCH_CHECK();
    }
  }
  if (splits > 1) return pc_topk_merge(ps, pi, rows, splits, k, out_scores, out_idx, stream);
  return PC_OK;
}

extern "C" size_t pc_topk_by_type_workspace_bytes(int64_t rows, int k, int splits) {
  if (rows <= 0) return 0;
  return align_up(size_t(rows) * 8, 256) + align_up(pc_sort_keys_workspace_bytes(rows), 256) + 2 * align_up(size_t(rows) * 4, 256) +
         pc_topk_groups_workspace_bytes(rows, k, splits);
}

extern "C" int pc_topk_by_type(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                               const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                               int64_t index_base, double* out_scores, int64_t* out_idx, void* workspace,
                               size_t workspace_bytes, pc_stream_t stream) {
  PC_REQUIRE(rows >= 0 && rows < (int64_t(1) << 31), PC_ERR_INVALID, "topk_by_type: bad row count");
  if (rows == 0) return PC_OK;
  PC_REQUIRE(q && catalog && type_offsets && out_scores && out_idx && workspace, PC_ERR_INVALID, "topk_by_type: null pointer");
  PC_REQUIRE(n_types >= 1 && n_types < (1 << 30), PC_ERR_INVALID, "topk_by_type: bad n_types=%d", n_types);
  PC_REQUIRE(k >= 1 && k <= PC_TOPK_MAX_K, PC_ERR_UNSUPPORTED, "topk_by_type: k=%d outside [1,%d]", k, PC_TOPK_MAX_K);
  PC_REQUIRE(dim >= DCH && dim % DCH == 0 && dim <= 1024, PC_ERR_UNSUPPORTED, "topk_by_type: dim=%d must be a multiple of %d (<= 1024)", dim, DCH);
  PC_REQUIRE(splits >= 1 && splits <= 65535, PC_ERR_UNSUPPORTED, "topk_by_type: bad splits");
  PC_REQUIRE(workspace_bytes >= pc_topk_by_type_workspace_bytes(rows, k, splits), PC_ERR_WORKSPACE, "topk_by_type: workspace too small");
  cudaStream_t st = as_stream(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  uint64_t* keys = reinterpret_cast<uint64_t*>(ws);             ws += align_up(size_t(rows) * 8, 256);
  void* sort_ws = ws;                                            const size_t sort_bytes = pc_sort_keys_workspace_bytes(rows);
  ws += align_up(sort_bytes, 256);
  int32_t* row_ids = reinterpret_cast<int32_t*>(ws);             ws += align_up(size_t(rows) * 4, 256);
  int32_t* grp_rows = reinterpret_cast<int32_t*>(ws);            ws += align_up(size_t(rows) * 4, 256);
  const unsigned tb = unsigned(ceil_div(rows, 256));
  type_keys_kernel<<<tb, 256, 0, st>>>(row_type, rows, n_types, keys);
  PC_LAUNCH_CHECK();
  // keys are created in ascending row order and the sort is stable: only the type bytes take part
  uint32_t mask = 0;
  for (int b = 0; b < 4; ++b)
    if ((uint64_t(n_types) >> (8 * b)) != 0) mask |= 1u << (4 + b);
  if (int rc = pc_sort_keys(keys, rows, mask, sort_ws, sort_bytes, stream)) return rc;
  double* ps = out_scores;
  int64_t* pi = out_idx;
  if (splits > 1) {
    ps = reinterpret_cast<double*>(ws);
    pi = reinterpret_cast<int64_t*>(ps + size_t(rows) * splits * k);
  }
  if (k > WARP_K) {
    if (int rc = by_type_large(q, rows, dim, catalog, members, type_offsets, n_types, keys, row_ids, grp_rows, k, splits,
                               index_base, ps, pi, st))
      return rc;
  } else {
    topk_plan_kernel<RB><<<tb, 256, 0, st>>>(keys, rows, row_ids, grp_rows);
    PC_LAUNCH_CHECK();
    const size_t smem = size_t(RB) * dim * sizeof(double) +
                        std::max(size_t(TK_WARPS) * 2 * TILE_FLOATS * sizeof(float), size_t(TK_WARPS) * RB * 32 * sizeof(Cand));
    PC_REQUIRE(smem <= 200 * 1024, PC_ERR_UNSUPPORTED, "topk_by_type: shared memory budget exceeded");
    PC_CUDA(cudaFuncSetAttribute(topk_planned_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    for (int64_t p0 = 0; p0 < rows; p0 += 65535) {   // gridDim.y limit
      const int64_t np = rows - p0 < 65535 ? rows - p0 : 65535;
      dim3 grid{unsigned(splits), unsigned(np), 1u};
      topk_planned_kernel<<<grid, TK_WARPS * 32, smem, st>>>(q, dim, catalog, members, row_ids, grp_rows, keys, type_offsets,
                                                             n_types, p0, k, splits, index_base, ps, pi);
      PC_LAUNCH_CHECK();
    }
  }
  if (splits > 1) return pc_topk_merge(ps, pi, rows, splits, k, out_scores, out_idx, stream);
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
  cudaStream_t st = as_stream(stream);
  double* ps = out_scores;
  int64_t* pi = out_idx;
  if (splits > 1) {
    PC_REQUIRE(workspace && workspace_bytes >= pc_topk_rows_workspace_bytes(rows, k, splits), PC_ERR_WORKSPACE,
               "topk_rows: workspace too small");
    ps = reinterpret_cast<double*>(workspace);
    pi = reinterpret_cast<int64_t*>(ps + size_t(rows) * splits * k);
  }
  for (int64_t r0 = 0; r0 < rows; r0 += 65535) {
    const int64_t nr = rows - r0 < 65535 ? rows - r0 : 65535;
    dim3 grid{unsigned(splits), unsigned(nr), 1u};
    if (k > WARP_K) {
      const int cap = large_cap(k, LK_STREAM_PASS);
      topk_values_large_kernel<<<grid, LK_THREADS, stream_smem_bytes(cap), st>>>(values + r0 * cols, cols, k, cap, splits,
                                                                                ps + r0 * splits * k, pi + r0 * splits * k);
    } else {
      topk_values_kernel<<<grid, TK_WARPS * 32, 0, st>>>(values + r0 * cols, cols, k, splits, ps + r0 * splits * k,
                                                         pi + r0 * splits * k);
    }
    PC_LAUNCH_CHECK();
  }
  if (splits > 1) return pc_topk_merge(ps, pi, rows, splits, k, out_scores, out_idx, stream);
  return PC_OK;
}
