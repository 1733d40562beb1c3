// Device-side negative sampling for the similarity (triplet) batches.
//
// Replaces SimilarityDataset._get_negative_samples of /root/reference/src/data/data_loader.py:27-40
// (per item: rebuild the anchor's similar set by scanning all pairs, then rejection-sample k products
// that are not the anchor, not similar to it and pairwise distinct).  Here the similar set is one CSR row
// (binary search) and every anchor is one thread with a counter-based generator, so a batch of negatives is
// one launch and is reproducible from (seed, batch slot) alone.
//
// pc_triplet_batch_rows then gathers the batch's feature rows (anchors, co-view neighbours, positives, negatives) for the
// graph-native training step, again in one launch.
#include "common.cuh"

namespace pc {
namespace {

__device__ __forceinline__ uint64_t splitmix(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void sample_negatives_kernel(const int32_t* __restrict__ anchor, const int64_t* __restrict__ sim_rowptr,
                                        const int32_t* __restrict__ sim_col, int64_t batch, int32_t n_nodes, int k,
                                        uint64_t seed, int32_t* __restrict__ out) {
  const int64_t b = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const int32_t a = anchor[b];
  const int64_t lo = sim_rowptr[a], hi = sim_rowptr[a + 1];
  int32_t* mine = out + b * k;
  uint64_t state = splitmix(seed ^ (uint64_t(b) * 0xD1B54A32D192ED03ull));
  int got = 0;
  const int max_attempts = 64 * k + 64;
  for (int attempt = 0; got < k && attempt < max_attempts; ++attempt) {
    state = splitmix(state);
    const int32_t c = int32_t((state >> 11) % uint64_t(n_nodes));   // uniform over products (random.choice, :34)
    bool ok = c != a;                                               // :35
    if (ok) {                                                       // :36  not in the anchor's similar set
      int64_t l = lo, h = hi;
      while (l < h) {
        const int64_t mid = (l + h) >> 1;
        if (sim_col[mid] < c) l = mid + 1; else h = mid;
      }
      ok = !(l < hi && sim_col[l] == c);
    }
    for (int j = 0; ok && j < got; ++j) ok = mine[j] != c;          // :37  distinct
    if (ok) mine[got++] = c;
  }
  // degenerate graphs (almost every product similar to the anchor): finish with a linear scan, never spin forever
  for (int32_t c = 0; got < k && c < n_nodes; ++c) {
    bool ok = c != a;
    if (ok) {
      int64_t l = lo, h = hi;
      while (l < h) {
        const int64_t mid = (l + h) >> 1;
        if (sim_col[mid] < c) l = mid + 1; else h = mid;
      }
      ok = !(l < hi && sim_col[l] == c);
    }
    for (int j = 0; ok && j < got; ++j) ok = mine[j] != c;
    if (ok) mine[got++] = c;
  }
  for (; got < k; ++got) mine[got] = -1;                            // fewer than k eligible products exist
}

// Feature rows of one triplet batch (the tensors collate_fn stacks, data_loader.py:171-206, without the padding).  One warp
// per anchor b walks its 2 + kneg + deg(b) rows - anchor, positive, negatives, then the co-view neighbours in CSR order - in
// chunks of 32: lane l resolves the (source, destination) row of slot l of the chunk (and writes the edge's batch slot),
// then the warp copies the chunk's rows four at a time, every row as coalesced float4 loads / stores.
__global__ void __launch_bounds__(256)
triplet_batch_rows_kernel(const float4* __restrict__ table, int64_t ld4, int width4, const int64_t* __restrict__ anchor,
                          const int64_t* __restrict__ positive, const int64_t* __restrict__ negatives, int64_t batch, int kneg,
                          const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                          const int64_t* __restrict__ nbr_ptr, int64_t n_nbr, float4* __restrict__ rows,
                          int32_t* __restrict__ edge_row) {
  const int64_t b = int64_t(blockIdx.x) * 8 + warp_id();
  if (b >= batch) return;
  const int lane = lane_id();
  const int64_t a = anchor[b];
  const int64_t src0 = rowptr[a], dst0 = nbr_ptr[b];
  const int64_t fixed = 2 + int64_t(kneg);
  const int64_t total = fixed + (nbr_ptr[b + 1] - dst0);
  const int64_t pos_row = batch + n_nbr + b, neg_row = 2 * batch + n_nbr + b * kneg;
  for (int64_t base = 0; base < total; base += 32) {
    const int64_t s = base + lane;
    int64_t src = 0, dst = 0;
    if (s < total) {
      if (s == 0) {
        src = a; dst = b;
      } else if (s == 1) {
        src = positive[b]; dst = pos_row;
      } else if (s < fixed) {
        src = negatives[b * kneg + (s - 2)]; dst = neg_row + (s - 2);
      } else {
        const int64_t e = s - fixed;
        src = col[src0 + e]; dst = batch + dst0 + e;
        edge_row[dst0 + e] = int32_t(b);
      }
    }
    const int m = int(total - base < 32 ? total - base : 32);
    int j = 0;
    for (; j + 4 <= m; j += 4) {
      const float4* s0 = table + __shfl_sync(0xffffffffu, src, j) * ld4;
      const float4* s1 = table + __shfl_sync(0xffffffffu, src, j + 1) * ld4;
      const float4* s2 = table + __shfl_sync(0xffffffffu, src, j + 2) * ld4;
      const float4* s3 = table + __shfl_sync(0xffffffffu, src, j + 3) * ld4;
      float4* d0 = rows + __shfl_sync(0xffffffffu, dst, j) * width4;
      float4* d1 = rows + __shfl_sync(0xffffffffu, dst, j + 1) * width4;
      float4* d2 = rows + __shfl_sync(0xffffffffu, dst, j + 2) * width4;
      float4* d3 = rows + __shfl_sync(0xffffffffu, dst, j + 3) * width4;
      for (int c = lane; c < width4; c += 32) {
        const float4 v0 = ldg4(s0 + c), v1 = ldg4(s1 + c), v2 = ldg4(s2 + c), v3 = ldg4(s3 + c);
        d0[c] = v0; d1[c] = v1; d2[c] = v2; d3[c] = v3;
      }
    }
    for (; j < m; ++j) {
      const float4* s0 = table + __shfl_sync(0xffffffffu, src, j) * ld4;
      float4* d0 = rows + __shfl_sync(0xffffffffu, dst, j) * width4;
      for (int c = lane; c < width4; c += 32) d0[c] = ldg4(s0 + c);
    }
  }
}

}  // namespace
}  // namespace pc

using namespace pc;

extern "C" int pc_sample_negatives(const int32_t* anchor, const int64_t* sim_rowptr, const int32_t* sim_col, int64_t batch,
                                   int32_t n_nodes, int k, uint64_t seed, int32_t* out, pc_stream_t stream) {
  PC_REQUIRE(batch >= 0 && n_nodes > 0 && k >= 1 && k <= 64, PC_ERR_INVALID, "sample_negatives: bad sizes");
  if (batch == 0) return PC_OK;
  PC_REQUIRE(anchor && sim_rowptr && out, PC_ERR_INVALID, "sample_negatives: null pointer");
  sample_negatives_kernel<<<unsigned(ceil_div(batch, 128)), 128, 0, as_stream(stream)>>>(anchor, sim_rowptr, sim_col, batch,
                                                                                      n_nodes, k, seed, out);
  PC_LAUNCH_CHECK();
  return PC_OK;
}

extern "C" int pc_triplet_batch_rows(const float* table, int64_t ld, int dim, const int64_t* anchor, const int64_t* positive,
                                     const int64_t* negatives, int64_t batch, int kneg, const int64_t* rowptr, const int32_t* col,
                                     const int64_t* nbr_ptr, int64_t n_nbr, float* rows, int32_t* edge_row, pc_stream_t stream) {
  PC_REQUIRE(dim > 0 && dim % 4 == 0 && dim <= 1024 && ld >= dim && ld % 4 == 0, PC_ERR_INVALID,
             "triplet_batch_rows: bad dim=%d ld=%lld", dim, (long long)ld);
  PC_REQUIRE(batch >= 0 && batch < (int64_t(1) << 31) && kneg >= 1 && n_nbr >= 0 && n_nbr < (int64_t(1) << 31),
             PC_ERR_INVALID, "triplet_batch_rows: bad sizes batch=%lld kneg=%d n_nbr=%lld", (long long)batch, kneg,
             (long long)n_nbr);
  if (batch == 0) return PC_OK;
  PC_REQUIRE(table && anchor && positive && negatives && rowptr && nbr_ptr && rows && (n_nbr == 0 || (col && edge_row)),
             PC_ERR_INVALID, "triplet_batch_rows: null pointer");
  PC_REQUIRE(reinterpret_cast<uintptr_t>(table) % 16 == 0 && reinterpret_cast<uintptr_t>(rows) % 16 == 0, PC_ERR_INVALID,
             "triplet_batch_rows: table and rows must be 16-byte aligned");
  triplet_batch_rows_kernel<<<unsigned(ceil_div(batch, 8)), 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const float4*>(table), ld / 4, dim / 4, anchor, positive, negatives, batch, kneg, rowptr, col, nbr_ptr,
      n_nbr, reinterpret_cast<float4*>(rows), edge_row);
  PC_LAUNCH_CHECK();
  return PC_OK;
}
