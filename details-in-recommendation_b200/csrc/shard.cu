// Row-sharded tables: the id-only kernels (keys, distinct-row numbering).
//
// Tables are sharded by row over G ranks (owner = global row mod G, local row = global row div G:
// modulo, so hot low-numbered rows spread evenly).  The batch stays data-parallel.  Per step a rank
//   1. dir_shard_keys[_sort]  forms one composite key per lookup, (owner, local row), owner-major, and sorts
//                             (key, lookup position)                                  [keys.cuh, embed_bwd.cu, radix.cuh]
//   2. dir_shard_unique       numbers the distinct keys: only those cross NVLink
//   3. the exchange: ids to the owners, rows back, per-distinct-row gradient sums to the owners -- stored
//      straight into the peers' buffers by the kernels of shard_peer.cu
//   4. dir_embed_fm_fwd       runs on the received unique-row buffer, indexed by `inv`  [embed_fwd.cu]
// Bags (CSR) take dir_shard_bag_keys instead of step 1's key kernel; everything after it is shared.
// The reference has no counterpart: its only hook is the partitioner wrapped around the embedding
// variables (models/DeepFM/deepFM.py:163-175), which under a TF parameter-server cluster shards
// variables by row and ships ids / IndexedSlices over gRPC.
#include "common.cuh"
#include "keys.cuh"

namespace dir {

__global__ void __launch_bounds__(256) shard_keys_kernel(const KeyArgs a, uint32_t* __restrict__ keys) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // entry of the [B, n_sel] key list
  if (o >= a.n) return;
  keys[o] = make_key(a, o);
}

// ------------------------------------------------------------------------------ numbering the distinct keys
// Three small kernels over tiles of kUTile sorted entries (the list lives in L2):
//   count   head flags (entry differs from its left neighbour and is not pruned) per tile
//   scan    one CTA: exclusive prefix of the tile counts
//   number  per tile: block scan of the flags on top of the tile's base -> uidx / ulocal / inv / owner_off
// (no per-entry prefix array goes through memory, no library scan).
constexpr int kURounds = 2;              // rounds of 32 consecutive entries per warp (small tiles: the numbering
                                        // kernel's scattered inv stores want many warps in flight)
constexpr int kUTile = 8 * kURounds * 32;  // 8 warps per CTA

// head flags of the kURounds rounds of one warp (round r = entries wbase + r * 32 + lane): bit `lane` of heads[r]
__device__ __forceinline__ void warp_head_flags(const uint32_t* __restrict__ keys, int64_t n, uint32_t pruned,
                                                int64_t wbase, int lane, uint32_t (&k)[kURounds], unsigned (&heads)[kURounds],
                                                uint32_t& kleft) {
  kleft = (wbase > 0 && wbase - 1 < n) ? __ldg(keys + wbase - 1) : 0u;  // (uniform over the warp)
#pragma unroll
  for (int r = 0; r < kURounds; ++r) {
    const int64_t i = wbase + r * 32 + lane;
    k[r] = i < n ? __ldg(keys + i) : pruned;
  }
  uint32_t prev_last = kleft;
#pragma unroll
  for (int r = 0; r < kURounds; ++r) {
    const int64_t i = wbase + r * 32 + lane;
    uint32_t kp = __shfl_up_sync(0xffffffffu, k[r], 1);
    if (lane == 0) kp = prev_last;
    heads[r] = __ballot_sync(0xffffffffu, i < n && k[r] != pruned && (i == 0 || k[r] != kp));
    prev_last = __shfl_sync(0xffffffffu, k[r], 31);
  }
}

__global__ void __launch_bounds__(256)
unique_count_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t pruned, uint32_t* __restrict__ tilecnt) {
  __shared__ uint32_t s_warp[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wbase = (int64_t)blockIdx.x * kUTile + w * (kURounds * 32);
  uint32_t k[kURounds], kleft;
  unsigned heads[kURounds];
  warp_head_flags(keys, n, pruned, wbase, lane, k, heads, kleft);
  uint32_t c = 0;
#pragma unroll
  for (int r = 0; r < kURounds; ++r) c += (uint32_t)__popc(heads[r]);
  if (lane == 0) s_warp[w] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) t += s_warp[ww];
    tilecnt[blockIdx.x] = t;
  }
}

// in place: tilecnt[t] <- distinct keys in the tiles before t.  One CTA; a thread owns up to 16 consecutive tiles, so
// up to 4 096 tiles (1 M entries) take one block scan.
__global__ void __launch_bounds__(256) unique_scan_kernel(uint32_t* __restrict__ tilecnt, int64_t tiles) {
  __shared__ uint32_t s_warp[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t per = (tiles + 255) / 256;
  const int C = (int)(per < 16 ? per : 16);
  uint32_t carry = 0;
  for (int64_t c0 = 0; c0 < tiles; c0 += (int64_t)256 * C) {
    const int64_t i0 = c0 + (int64_t)threadIdx.x * C;
    uint32_t v[16];
    uint32_t sum = 0;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      v[e] = (e < C && i0 + e < tiles) ? tilecnt[i0 + e] : 0u;
      sum += v[e];
    }
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) {
      const uint32_t c = s_warp[ww];
      if (ww < w) base += c;
      tot += c;
    }
    __syncthreads();
    uint32_t run = carry + base + inc - sum;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      if (e < C && i0 + e < tiles) {
        tilecnt[i0 + e] = run;
        run += v[e];
      }
    }
    carry += tot;
  }
}

// Numbers the distinct keys of the sorted list and, where the owner changes between two neighbouring entries,
// writes owner_off[g] = number of distinct keys below g * cap for every g in between (g = 0..G; every g is written
// exactly once because the owners are non-decreasing).
__global__ void __launch_bounds__(256)
shard_number_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ pos,
                    const uint32_t* __restrict__ tilebase, int64_t n, uint32_t pruned, uint32_t cap, int G,
                    const int32_t* __restrict__ field_sel, int n_sel, int F,
                    uint32_t* __restrict__ uidx, int32_t* __restrict__ ulocal,
                    int64_t* __restrict__ inv, int64_t* __restrict__ owner_off) {
  __shared__ uint32_t s_warp[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wbase = (int64_t)blockIdx.x * kUTile + w * (kURounds * 32);
  uint32_t k[kURounds], kleft;
  unsigned heads[kURounds];
  warp_head_flags(keys, n, pruned, wbase, lane, k, heads, kleft);
  uint32_t c = 0;
#pragma unroll
  for (int r = 0; r < kURounds; ++r) c += (uint32_t)__popc(heads[r]);
  if (lane == 0) s_warp[w] = c;
  __syncthreads();
  uint32_t run = __ldg(tilebase + blockIdx.x);  // distinct keys before this warp's first entry
#pragma unroll
  for (int ww = 0; ww < 8; ++ww)
    if (ww < w) run += s_warp[ww];
  uint32_t prev_last = kleft;
#pragma unroll
  for (int r = 0; r < kURounds; ++r) {
    const int64_t i = wbase + r * 32 + lane;
    uint32_t kp = __shfl_up_sync(0xffffffffu, k[r], 1);
    if (lane == 0) kp = prev_last;
    prev_last = __shfl_sync(0xffffffffu, k[r], 31);
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t before = run + (uint32_t)__popc(heads[r] & lt);  // distinct keys before entry i
    const bool head = (heads[r] >> lane) & 1u;
    const uint32_t incl = before + (head ? 1u : 0u);
    run += (uint32_t)__popc(heads[r]);
    if (i >= n) continue;
    const uint32_t kk = k[r];
    {
      const int o_cur = (int)(kk / cap);  // G for a pruned entry
      const int o_prev = i > 0 ? (int)(kp / cap) : -1;
      if (o_cur != o_prev)
        for (int g = o_prev + 1; g <= o_cur && g <= G; ++g) owner_off[g] = (int64_t)before;
      if (i == n - 1)
        for (int g = o_cur + 1; g <= G; ++g) owner_off[g] = (int64_t)incl;
    }
    uint32_t p = __ldg(pos + i);
    if (field_sel != nullptr) {  // entry of the compact [B, n_sel] list -> position in the [B, F] inputs
      const uint32_t b = p / (uint32_t)n_sel;
      p = b * (uint32_t)F + (uint32_t)__ldg(field_sel + (p - b * (uint32_t)n_sel));
    }
    if (kk == pruned) {
      uidx[i] = 0u;
      if (inv) inv[p] = -1;  // pruned by the forward kernel (id < 0)
    } else {
      const uint32_t u = incl - 1u;
      uidx[i] = u;
      if (inv) inv[p] = (int64_t)u;
      if (head) ulocal[u] = (int32_t)(kk % cap);
    }
  }
}

// Bags (CSR): one thread per (sample, field) slot walks its entries; entry j gets the composite key of its row,
// or the pruned key (id < 0, weight <= 0, id beyond the field: the last also raises oob_flag).
__global__ void __launch_bounds__(256)
shard_bag_keys_kernel(const int64_t* __restrict__ bag_offsets, const int64_t* __restrict__ bag_index,
                      const float* __restrict__ bag_weight, const int64_t* __restrict__ field_offset,
                      const int64_t* __restrict__ field_rows, int64_t n_rows, int64_t n_slots, int F, int G,
                      int64_t cap, uint32_t* __restrict__ keys, int* oob_flag) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int f = (int)(s % F);
  const int64_t lo = __ldg(field_offset + f);
  const int64_t nf = field_rows ? __ldg(field_rows + f) : n_rows - lo;
  const int64_t j1 = __ldg(bag_offsets + s + 1);
  for (int64_t j = __ldg(bag_offsets + s); j < j1; ++j) {
    const int64_t id = __ldg(bag_index + j);
    const float wv = bag_weight ? __ldg(bag_weight + j) : 1.f;
    bool keep = id >= 0 && wv > 0.f;
    if (keep && id >= nf) {
      keep = false;
      if (oob_flag) *oob_flag = 1;
    }
    const uint32_t row = (uint32_t)(lo + id);
    uint32_t key = row;
    if (G > 1) key = (row % (uint32_t)G) * (uint32_t)cap + row / (uint32_t)G;
    keys[j] = keep ? key : (uint32_t)(G * cap);
  }
}

struct UniqueWs {
  uint32_t* tilecnt;  // [tiles] head flags per tile, then their exclusive prefix
  int64_t tiles;
  size_t total;
};

static UniqueWs unique_carve(void* base, int64_t n) {
  UniqueWs w;
  w.tiles = (n + kUTile - 1) / kUTile;
  w.tilecnt = reinterpret_cast<uint32_t*>(base);
  w.total = align_up((size_t)w.tiles * 4, 256);
  return w;
}

}  // namespace dir

extern "C" int dir_shard_keys(const int64_t* feature_index, const float* feature_value,
                              const int64_t* field_offset, const int64_t* field_rows,
                              int64_t n_rows, int64_t B, int F, int G, const int32_t* field_sel,
                              int n_sel, uint32_t* keys, int* oob_flag, dir_stream_t stream) {
  using namespace dir;
  KeyArgs a;
  if (int rc = key_args("shard_keys", feature_index, feature_value, field_offset, field_rows, n_rows, B, F, G,
                        field_sel, n_sel, oob_flag, a))
    return rc;
  if (a.n == 0) return 0;
  if (!keys) return fail(DIR_EINVAL, "shard_keys: null pointer");
  shard_keys_kernel<<<(unsigned)((a.n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, keys);
  return launched("shard_keys");
}

extern "C" int dir_shard_bag_keys(const int64_t* bag_offsets, const int64_t* bag_index, const float* bag_weight,
                                  int64_t nnz, const int64_t* field_offset, const int64_t* field_rows,
                                  int64_t n_rows, int64_t B, int F, int G, uint32_t* keys, int* oob_flag,
                                  dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0 || G <= 0 || n_rows <= 0 || nnz < 0 || nnz >= 0x7fffffffLL)
    return fail(DIR_EINVAL, "shard_bag_keys: B >= 0, F > 0, G > 0, n_rows > 0, 0 <= nnz < 2^31 required");
  const int64_t cap = (n_rows + G - 1) / G;
  if ((uint64_t)cap * (uint64_t)G >= 0xffffffffULL)
    return fail(DIR_EINVAL, "shard_bag_keys: ceil(n_rows / G) * G must be < 2^32-1");
  if (B * F >= 0x7fffffffLL) return fail(DIR_EINVAL, "shard_bag_keys: B*F must be < 2^31");
  if (B == 0 || nnz == 0) return 0;
  if (!bag_offsets || !bag_index || !field_offset || !keys) return fail(DIR_EINVAL, "shard_bag_keys: null pointer");
  shard_bag_keys_kernel<<<(unsigned)((B * F + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      bag_offsets, bag_index, bag_weight, field_offset, field_rows, n_rows, B * F, F, G, cap, keys, oob_flag);
  return launched("shard_bag_keys");
}

extern "C" size_t dir_shard_unique_workspace_bytes(int64_t n_lookups) {
  if (n_lookups <= 0) return 0;
  return dir::unique_carve(nullptr, n_lookups).total;
}

extern "C" int dir_shard_unique(const uint32_t* sorted_keys, const uint32_t* sorted_pos,
                                int64_t n_lookups, int64_t n_rows, int G, const int32_t* field_sel, int n_sel,
                                int F, uint32_t* uidx, int32_t* unique_local_rows, int64_t* inv,
                                int64_t* owner_off, void* workspace, size_t workspace_bytes,
                                dir_stream_t stream) {
  using namespace dir;
  if (n_lookups < 0 || n_lookups >= 0x7fffffffLL || G <= 0 || G > 1023 || n_rows <= 0)
    return fail(DIR_EINVAL, "shard_unique: 0 <= n_lookups < 2^31, 0 < G <= 1023, n_rows > 0 required");
  if (!owner_off) return fail(DIR_EINVAL, "shard_unique: owner_off is required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_lookups == 0) {
    cudaMemsetAsync(owner_off, 0, (size_t)(G + 1) * 8, st);
    return 0;
  }
  if (!sorted_keys || !sorted_pos || !uidx || !unique_local_rows || !workspace)
    return fail(DIR_EINVAL, "shard_unique: null pointer");
  if (field_sel != nullptr && (n_sel <= 0 || n_sel > F || n_lookups % n_sel != 0))
    return fail(DIR_EINVAL, "shard_unique: with field_sel, 0 < n_sel <= F and n_lookups = B * n_sel are required");
  const int64_t cap = (n_rows + G - 1) / G;
  const uint32_t pruned = (uint32_t)(cap * G);
  UniqueWs w = unique_carve(workspace, n_lookups);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "shard_unique: workspace too small");
  unique_count_kernel<<<(unsigned)w.tiles, 256, 0, st>>>(sorted_keys, n_lookups, pruned, w.tilecnt);
  unique_scan_kernel<<<1, 256, 0, st>>>(w.tilecnt, w.tiles);
  shard_number_kernel<<<(unsigned)w.tiles, 256, 0, st>>>(
      sorted_keys, sorted_pos, w.tilecnt, n_lookups, pruned, (uint32_t)cap, G, field_sel, n_sel, F, uidx,
      unique_local_rows, inv, owner_off);
  return launched("shard_unique", 3);
}

// ------------------------------------------------------------------------------------------------
// Tables too large to come from the host (cfg4: 880 M rows) are filled on the device from a counter hash,
// so that any row can be reproduced without the table (oracle/deepctr_oracle.py: counter_rows).
namespace dir {
__host__ __device__ inline uint64_t mix64(uint64_t x) {  // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void __launch_bounds__(256)
table_init_counter_kernel(float* __restrict__ table, int64_t row_stride, int64_t n_local, int K, int G, int rank,
                          int64_t n_rows, uint64_t seed, float scale) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = t / K;
  const int k = (int)(t % K);
  if (i >= n_local) return;
  const int64_t row = i * G + rank;
  float v = 0.f;
  if (row < n_rows) {
    const uint64_t h = mix64(seed ^ mix64((uint64_t)row * 64ull + (uint64_t)k));
    // four 16-bit uniforms: the sum is an integer in [0, 4 * 65535], centred exactly, scaled by one multiply
    const int sum = (int)(h & 0xffff) + (int)((h >> 16) & 0xffff) + (int)((h >> 32) & 0xffff) + (int)(h >> 48);
    v = __fmul_rn((float)(sum - 131070), scale);
  }
  table[i * row_stride + k] = v;
}
}  // namespace dir

extern "C" int dir_table_init_counter(float* table, int64_t row_stride, int64_t n_local_rows, int K, int G,
                                      int rank, int64_t n_rows, uint64_t seed, float sd, dir_stream_t stream) {
  using namespace dir;
  if (!table || n_local_rows <= 0 || K <= 0 || K > 64 || G <= 0 || rank < 0 || rank >= G || row_stride < K)
    return fail(DIR_EINVAL, "table_init_counter: table, n_local_rows > 0, 0 < K <= 64 <= row_stride, 0 <= rank < G required");
  // a 16-bit uniform has variance (65536^2 - 1) / 12; four of them: sd_sum = sqrt((65536^2 - 1) / 3)
  const float scale = sd / 37837.2272f;
  const int64_t n = n_local_rows * K;
  const int64_t grid = (n + 255) / 256;
  if (grid > 0x7fffffffLL) return fail(DIR_EINVAL, "table_init_counter: table too large for one launch");
  table_init_counter_kernel<<<(unsigned)grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      table, row_stride, n_local_rows, K, G, rank, n_rows, seed, scale);
  return launched("table_init_counter");
}
