// Row-sharded tables, device-driven exchange over NVLink peer memory (no NCCL, no host read on the step).
//
// Every rank owns one exchange buffer per parity with the same layout (dir_peer_layout); peers store
// straight into it through peer-mapped addresses.  Sizes that depend on the data travel as headers and are
// read on the device, so every launch of a step is sized by capacities known up front and the whole step --
// id phase included -- can be replayed from a CUDA graph:
//
//   requester q                                         owner o
//   dir_shard_keys / sort / dir_shard_unique  (ids only)
//   dir_shard_ids_push    hdr[q] = (count, base_u), ids[q][0..count)  -->  o's buffer
//   ---- barrier (ids) ----
//                                                       dir_shard_slots      slot[row][q] = i + 1
//                                                       dir_shard_gather_send  T[row] -> q's rows[base_u + i],
//                                                                              w[row] -> q's w[base_u + i]
//   ---- barrier (rows) ----
//   dir_embed_fm_fwd on rows / w, indexed by inv
//   dir_embed_bwd_reduce_emit_to   per-distinct-row sums  -->  o's g[q][i]       (embed_bwd.cu)
//   dir_shard_g1_push              first-order sums       -->  o's g1[q][i]
//   dir_shard_dense_emit           one-row fields' sums   -->  everybody's dense[q][j]
//   ---- barrier (grads) ----
//                                                       dir_shard_owner_update  per local row: the requesters'
//                                                         sums added in rank order, fused row update
//                                                       dir_shard_slots(clear)
//   dir_shard_dense_apply   replicated one-row fields: ranks' sums added in rank order, same update everywhere
//
// With clip_norm (tf.clip_by_norm per column), the owner half after the grads barrier is instead
//                                                       dir_shard_owner_sqnorms  per column: squares of the merged
//                                                         sums -> norm[me] of every rank's norm buffer
//   ---- barrier (norms) ----
//                                                       dir_shard_owner_update_clipped  partials combined in rank
//                                                         order, the same update with each sum scaled
//   dir_shard_dense_apply_clipped   replicated one-row fields, each clipped by its own sum
//
// With optimizer='adam' (TF's Adam decays every row's moments), the owner half after the grads barrier (and, with a
// clip, the norm pass and its barrier) is one sweep; every field goes through the exchange (no replicated rows)
//                                                       dir_shard_owner_apply_adam  every local row decayed, the
//                                                         requesters' sums merged in rank order where a row has them
//
// The owner never sorts: a requester sends each row at most once, so slot[row][q] (one cell per local row and
// requester, written without atomics) tells an arrival whether an earlier rank asked for the same row; the first
// one merges.  Deterministic: no floating-point atomics, sums in rank order.  A cell is (epoch << 24) | (i + 1) and
// counts only while its epoch is the buffer's current one, so nothing has to be cleared after a step; the epoch
// (1..255, advanced on the device by the id push) wraps once per 255 uses, when the whole map is zeroed.
//
// Reference: the partitioner hook around the embedding variables, models/DeepFM/deepFM.py:163-175 (under a TF
// parameter-server cluster the variables are sharded by row and ids / IndexedSlices travel over gRPC).
#include "adam.cuh"

namespace dir {

constexpr int kMaxG = 64;
constexpr int kPeerCtas = kSMs * 8;  // grid-stride launches: the real counts are known on the device only

__device__ __forceinline__ char* peer_buf(const dir_peer_layout& L, int q) {
  return reinterpret_cast<char*>(__ldg(L.peer_base + q));
}
__device__ __forceinline__ int seg_of(const int64_t* s, int G, int64_t i) {  // s[G+1] ascending, in shared memory
  int q = 0;
  while (q + 1 < G && i >= s[q + 1]) ++q;
  return q;
}

// requester: header + distinct local rows to every owner
__global__ void __launch_bounds__(256)
peer_ids_push_kernel(const dir_peer_layout L, const int32_t* __restrict__ ulocal,
                     const int64_t* __restrict__ owner_off, int64_t n_cap, int* err, uint32_t* epoch) {
  __shared__ int64_t s_off[kMaxG + 1];
  if (threadIdx.x <= L.G) s_off[threadIdx.x] = owner_off[threadIdx.x];
  if (epoch != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    // this buffer's slot map enters a new epoch: epoch[0] = current (1..255), epoch[1] = "zero the map first"
    const uint32_t e = epoch[0];
    epoch[1] = e >= 255u ? 1u : 0u;
    epoch[0] = e >= 255u ? 1u : e + 1u;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x < L.G) {
    const int o = threadIdx.x;
    int64_t cnt = s_off[o + 1] - s_off[o];
    if (cnt > L.seg_cap || s_off[L.G] > L.u_cap) {
      *err = 1;  // more distinct rows than the buffers were sized for: nothing is written out of bounds
      cnt = cnt > L.seg_cap ? L.seg_cap : cnt;
    }
    int64_t* hdr = reinterpret_cast<int64_t*>(peer_buf(L, o) + L.off_hdr) + (int64_t)L.rank * 4;
    hdr[0] = cnt;
    hdr[1] = s_off[o];
  }
  int64_t total = s_off[L.G];
  total = total < n_cap ? total : n_cap;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
    const int o = seg_of(s_off, L.G, i);
    const int64_t j = i - s_off[o];
    if (j < L.seg_cap)
      reinterpret_cast<int32_t*>(peer_buf(L, o) + L.off_ids)[(int64_t)L.rank * L.seg_cap + j] = __ldg(ulocal + i);
  }
}

// owner: what arrived.  pre[q] = arrivals from requesters < q; base[q] = where q keeps my rows.
struct Arrivals {
  int64_t pre[kMaxG + 1];
  int64_t base[kMaxG];
};
__device__ __forceinline__ void load_arrivals(const dir_peer_layout& L, Arrivals& s) {
  if (threadIdx.x == 0) {
    const int64_t* hdr = reinterpret_cast<const int64_t*>(L.local + L.off_hdr);
    int64_t pre = 0;
    for (int q = 0; q < L.G; ++q) {
      s.pre[q] = pre;
      int64_t c = hdr[q * 4];
      c = c < 0 ? 0 : (c > L.seg_cap ? L.seg_cap : c);
      pre += c;
      s.base[q] = hdr[q * 4 + 1];
    }
    s.pre[L.G] = pre;
  }
  __syncthreads();
}

// owner: the slot map is zeroed when its epoch wraps (epoch[1] set by the id push): a launch that exits at once
// 254 times out of 255
__global__ void __launch_bounds__(256)
peer_slots_reset_kernel(uint32_t* __restrict__ slot, int64_t n_cells, const uint32_t* __restrict__ epoch) {
  if (epoch[1] == 0u) return;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cells; i += step) slot[i] = 0u;
}

// owner: slot[row * G + q] = (epoch << 24) | (i + 1) for arrival i of requester q
__global__ void __launch_bounds__(256)
peer_slots_kernel(const dir_peer_layout L, uint32_t* __restrict__ slot, int64_t n_local, int* err,
                  int64_t* zero_counter, const uint32_t* __restrict__ epoch) {
  __shared__ Arrivals s;
  if (zero_counter != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero_counter = 0;
  load_arrivals(L, s);
  const uint32_t tag = epoch[0] << 24;
  const int32_t* ids = reinterpret_cast<const int32_t*>(L.local + L.off_ids);
  const int64_t total = s.pre[L.G];
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < total; a += step) {
    const int q = seg_of(s.pre, L.G, a);
    const int64_t i = a - s.pre[q];
    const int64_t r = __ldg(ids + (int64_t)q * L.seg_cap + i);
    if (r < 0 || r >= n_local) {
      *err = 2;
      continue;
    }
    slot[r * L.G + q] = tag | (uint32_t)(i + 1);
  }
}

// owner: fused gather + send.  The arrivals are cut into tiles of 256 consecutive arrivals of one requester
// (16 KB of contiguous destination rows); a CTA takes tiles t = blockIdx.x, + gridDim.x, ... where tile t belongs to
// requester (rank + 1 + t) mod G: every destination is being written all the time, and no two ranks start on the
// same one (processing requester 0's rows first on every rank makes rank 0's NVLink ingress the bottleneck for all
// of them).  LPR lanes carry one row (16 bytes each); a thread has up to four row loads in flight before its first
// NVLink store.  The first-order weights of the tile go out lane-per-arrival (128-byte contiguous stores per warp).
// CTA 0 also refreshes the replicated one-row fields' rows behind this rank's own rows.
constexpr int kTileArr = 256;
template <int LPR>
__global__ void __launch_bounds__(256)
peer_gather_send_kernel(const dir_peer_layout L, const float* __restrict__ table, int64_t row_stride,
                        const float* __restrict__ lin, int64_t lin_stride,
                        const float* __restrict__ dense_table, int64_t dense_stride,
                        const float* __restrict__ dense_lin) {
  constexpr int K = LPR * 4;
  constexpr int UN = LPR < 4 ? LPR : 4;  // row loads in flight per thread
  __shared__ Arrivals s;
  __shared__ char* s_peer[kMaxG];
  __shared__ int64_t s_tiles;
  if (threadIdx.x < L.G) s_peer[threadIdx.x] = peer_buf(L, threadIdx.x);
  load_arrivals(L, s);
  if (threadIdx.x == 0) {
    int64_t m = 0;
    for (int q = 0; q < L.G; ++q) {
      const int64_t c = (s.pre[q + 1] - s.pre[q] + kTileArr - 1) / kTileArr;
      m = c > m ? c : m;
    }
    s_tiles = m;
  }
  __syncthreads();
  const int32_t* ids = reinterpret_cast<const int32_t*>(L.local + L.off_ids);
  const int G = L.G;
  const int64_t T = s_tiles * G;
  for (int64_t t = blockIdx.x; t < T; t += gridDim.x) {
    const int q = (int)((L.rank + 1 + t % G) % G);
    const int64_t i0 = (t / G) * kTileArr;
    const int64_t cnt = s.pre[q + 1] - s.pre[q];
    if (i0 >= cnt) continue;
    const int n = (int)(cnt - i0 < kTileArr ? cnt - i0 : kTileArr);
    const int32_t* tid_ids = ids + (int64_t)q * L.seg_cap + i0;
    const int64_t d0 = s.base[q] + i0;  // first destination row of the tile
    if (d0 < 0 || d0 + n > L.u_cap) continue;
    float4* drows = reinterpret_cast<float4*>(s_peer[q] + L.off_rows) + d0 * LPR;
#pragma unroll
    for (int k0 = 0; k0 < LPR; k0 += UN) {
      int64_t r[UN];
      int e[UN];
      float4 v[UN];
#pragma unroll
      for (int k = 0; k < UN; ++k) {
        e[k] = threadIdx.x + 256 * (k0 + k);  // float4 of the tile: arrival e / LPR, part e % LPR
        r[k] = e[k] / LPR < n ? (int64_t)__ldg(tid_ids + e[k] / LPR) : -1;
      }
#pragma unroll
      for (int k = 0; k < UN; ++k)
        if (r[k] >= 0) v[k] = __ldg(reinterpret_cast<const float4*>(table + r[k] * row_stride) + e[k] % LPR);
#pragma unroll
      for (int k = 0; k < UN; ++k)
        if (r[k] >= 0) drows[e[k]] = v[k];
    }
    if (lin != nullptr && (int)threadIdx.x < n)
      reinterpret_cast<float*>(s_peer[q] + L.off_w)[d0 + threadIdx.x] =
          __ldg(lin + (int64_t)__ldg(tid_ids + threadIdx.x) * lin_stride);
  }
  if (blockIdx.x == 0 && L.n_dense > 0 && dense_table != nullptr) {
    float* rows = reinterpret_cast<float*>(L.local + L.off_rows) + L.u_cap * K;
    float* w = reinterpret_cast<float*>(L.local + L.off_w) + L.u_cap;
    for (int e = threadIdx.x; e < L.n_dense * K; e += blockDim.x)
      rows[e] = dense_table[(int64_t)(e / K) * dense_stride + (e % K)];
    for (int j = threadIdx.x; j < L.n_dense; j += blockDim.x) w[j] = dense_lin ? dense_lin[j] : 0.f;
  }
}

// requester: first-order gradient sums of the distinct rows (g1_local[u], grouped by owner) -> owners
__global__ void __launch_bounds__(256)
peer_g1_push_kernel(const dir_peer_layout L, const float* __restrict__ g1_local,
                    const int64_t* __restrict__ owner_off, int64_t n_cap) {
  __shared__ int64_t s_off[kMaxG + 1];
  if (threadIdx.x <= L.G) s_off[threadIdx.x] = owner_off[threadIdx.x];
  __syncthreads();
  int64_t total = s_off[L.G];
  total = total < n_cap ? total : n_cap;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
    const int o = seg_of(s_off, L.G, i);
    const int64_t j = i - s_off[o];
    if (j < L.seg_cap)
      reinterpret_cast<float*>(peer_buf(L, o) + L.off_g1)[(int64_t)L.rank * L.seg_cap + j] = __ldg(g1_local + i);
  }
}

// owner: merge + fused update.  A warp takes 32 arrivals at a time.  Lane-per-arrival stage: local row, then the
// row's slot cells -- does an earlier requester merge this row (then this arrival has nothing to do), which later
// ones contribute.  Vector stage over the arrivals that lead, compacted: LPR lanes per row, the row / accumulator /
// gradient loads of PB passes in flight together; the other requesters' sums are added in a fixed order, then the
// fused update (row and accumulator share a 128-byte line).
// NBUF = 2: the batch was exchanged as two micro-batches, each through an exchange buffer (and slot map) of its own;
// half s of rank q counts as virtual requester s * G + q, and the merge runs over both buffers in that order.
struct OwnerSrc {
  const char* local[2];      // the exchange buffers (same layout)
  const uint32_t* slot[2];
  const uint32_t* epoch[2];
};

// CLIP: tf.clip_by_norm per column of the merged sums (dir_shard_owner_update_clipped).  The column's denominators come
// from the combined partials (clip.part, [F][kClipSlices][2]) into shared memory; a row's column is looked up from its
// local row (clip.field_offset: the columns' first local rows, ascending).
struct OwnerClip {
  const int64_t* field_offset;
  const double* part;
  int F;
  float clip;
};
// 16 KB, allocated only by the kernels that call it (an extern __shared__ array would add to every kernel's static
// shared memory in this file)
struct ClipSmem {
  int64_t off[kClipMaxFields];
  float den[kClipMaxFields], den1[kClipMaxFields];
};
__device__ __forceinline__ ClipSmem& clip_smem() {
  __shared__ ClipSmem cs;
  return cs;
}

template <int LPR, int NBUF, bool CLIP = false>
__global__ void __launch_bounds__(256, LPR <= 4 ? 3 : 1)
peer_owner_update_kernel(const dir_peer_layout L, const OwnerSrc src, float* table, float* accum,
                         int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride, const LinOpt lo,
                         const RowRule rule, int64_t n_local, unsigned long long* n_unique, const OwnerClip clip) {
  constexpr int SLOTS = 32 / LPR;
  constexpr int PB = LPR <= 4 ? 2 : 1;
  constexpr unsigned FULL = 0xffffffffu;
  __shared__ Arrivals s[NBUF];
  const int64_t* c_off = nullptr;
  const float *c_den = nullptr, *c_den1 = nullptr;
  if constexpr (CLIP) {
    ClipSmem& cs = clip_smem();
    clip_denominators(clip.part, clip.field_offset, clip.F, clip.clip, cs.off, cs.den, cs.den1);
    c_off = cs.off;
    c_den = cs.den;
    c_den1 = cs.den1;
  }
  uint32_t tag[NBUF];
  int64_t tot[NBUF];
#pragma unroll
  for (int b = 0; b < NBUF; ++b) {
    dir_peer_layout Lb = L;
    Lb.local = const_cast<char*>(src.local[b]);
    load_arrivals(Lb, s[b]);
    tag[b] = src.epoch[b][0];  // a cell counts only while it carries its buffer's current epoch
    tot[b] = s[b].pre[L.G];
  }
  const int64_t total = tot[0] + (NBUF > 1 ? tot[NBUF - 1] : 0);
  const bool adagrad = rule.opt != DIR_OPT_SGD;  // the rule keeps an accumulator
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR, grp = lane / LPR;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t pol_row = policy_evict_first();
  const int G = L.G;
  unsigned long long leaders = 0;
  for (int64_t a0 = warp * 32; a0 < total; a0 += nwarps * 32) {  // warp-uniform trip count
    // ---- lane-per-arrival stage
    int64_t a = a0 + lane;
    bool lead = false;
    int64_t e = 0, r = 0;        // e: this arrival's entry of gbuf / g1buf, + (buffer << 40)
    unsigned long long more = 0; // virtual requesters after this one that asked for the same row
    if (a < total) {
      const int b = (NBUF > 1 && a >= tot[0]) ? 1 : 0;
      if (b) a -= tot[0];
      const int q = seg_of(s[b].pre, G, a);
      const int64_t i = a - s[b].pre[q];
      e = (int64_t)q * L.seg_cap + i;
      r = __ldg(reinterpret_cast<const int32_t*>(src.local[b] + L.off_ids) + e);
      e |= (int64_t)b << 40;
      if (r >= 0 && r < n_local) {
        bool earlier = false;
#pragma unroll
        for (int bb = 0; bb < NBUF; ++bb) {
          const uint32_t* sl = src.slot[bb] + r * G;
          uint32_t sv[8];
#pragma unroll
          for (int p = 0; p < 8; ++p) sv[p] = p < G ? __ldg(sl + p) : 0u;  // independent loads, one sector
#pragma unroll
          for (int p = 0; p < 8; ++p) {
            const bool on = (sv[p] >> 24) == tag[bb];
            const int v = bb * G + p, me = b * G + q;
            earlier |= on && v < me;
            if (on && v > me) more |= 1ull << v;
          }
          for (int p = 8; p < G; ++p) {
            const bool on = (__ldg(sl + p) >> 24) == tag[bb];
            const int v = bb * G + p, me = b * G + q;
            earlier |= on && v < me;
            if (on && v > me) more |= 1ull << v;
          }
        }
        lead = !earlier;  // else an earlier (virtual) requester merges this row
      }
    }
    const unsigned lm = __ballot_sync(FULL, lead);
    const int nl = __popc(lm);
    leaders += (unsigned long long)nl;
    // ---- vector stage over the leading arrivals
    for (int k0 = 0; k0 < nl; k0 += SLOTS * PB) {
      int64_t rr[PB], ee[PB];
      unsigned long long mm[PB];
      bool on[PB];
      float4 T[PB], A[PB], g[PB];
      float g1[PB], w1[PB], n1[PB], z1[PB];
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const int n = k0 + j * SLOTS + grp;
        on[j] = n < nl;
        const int from = on[j] ? (int)__fns(lm, 0, n + 1) : 0;
        rr[j] = __shfl_sync(FULL, r, from);
        ee[j] = __shfl_sync(FULL, e, from);
        mm[j] = __shfl_sync(FULL, more, from);
        T[j] = A[j] = g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        g1[j] = w1[j] = n1[j] = z1[j] = 0.f;
        if (on[j]) {
          const int64_t ro = rr[j] * row_stride;
          T[j] = ld_hint(table + ro + sub * 4, pol_row);
          if (adagrad) A[j] = ld_hint(accum + ro + sub * 4, pol_row);
          const char* base = src.local[NBUF > 1 ? (int)(ee[j] >> 40) : 0];
          const int64_t ent = ee[j] & ((1ll << 40) - 1);
          g[j] = __ldg(reinterpret_cast<const float4*>(base + L.off_g) + ent * LPR + sub);
          if (sub == 0 && lin != nullptr) {
            g1[j] = __ldg(reinterpret_cast<const float*>(base + L.off_g1) + ent);
            w1[j] = lin[rr[j] * lin_stride];
            lin_load(lo, lin_accum, rr[j] * lin_stride, n1[j], z1[j]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        if (!on[j]) continue;
        unsigned long long m = mm[j];
        while (m) {  // fixed order: buffer, then rank
          const int v = __ffsll((long long)m) - 1;
          m &= m - 1;
          const int bb = NBUF > 1 ? v / G : 0, p = NBUF > 1 ? v - bb * G : v;
          const uint32_t sp = __ldg(src.slot[bb] + rr[j] * G + p) & 0xffffffu;
          const int64_t e2 = (int64_t)p * L.seg_cap + (sp - 1u);
          const float4 o = __ldg(reinterpret_cast<const float4*>(src.local[bb] + L.off_g) + e2 * LPR + sub);
          g[j].x = __fadd_rn(g[j].x, o.x);
          g[j].y = __fadd_rn(g[j].y, o.y);
          g[j].z = __fadd_rn(g[j].z, o.z);
          g[j].w = __fadd_rn(g[j].w, o.w);
          if (sub == 0 && lin != nullptr)
            g1[j] = __fadd_rn(g1[j], __ldg(reinterpret_cast<const float*>(src.local[bb] + L.off_g1) + e2));
        }
        if constexpr (CLIP) {
          int f = 0, hi = clip.F;  // last column whose first local row <= the row
          while (hi - f > 1) {
            const int mid = (f + hi) >> 1;
            if (c_off[mid] <= rr[j]) f = mid; else hi = mid;
          }
          g[j].x = clip1(g[j].x, clip.clip, c_den[f]);
          g[j].y = clip1(g[j].y, clip.clip, c_den[f]);
          g[j].z = clip1(g[j].z, clip.clip, c_den[f]);
          g[j].w = clip1(g[j].w, clip.clip, c_den[f]);
          g1[j] = clip1(g1[j], clip.clip, c_den1[f]);
        }
        const int64_t ro = rr[j] * row_stride;
        T[j].x = upd_rule(T[j].x, g[j].x, A[j].x, rule);
        T[j].y = upd_rule(T[j].y, g[j].y, A[j].y, rule);
        T[j].z = upd_rule(T[j].z, g[j].z, A[j].z, rule);
        T[j].w = upd_rule(T[j].w, g[j].w, A[j].w, rule);
        *(reinterpret_cast<float4*>(table + ro) + sub) = T[j];
        if (adagrad) *(reinterpret_cast<float4*>(accum + ro) + sub) = A[j];
        if (lin != nullptr && sub == 0) {
          const int64_t off = rr[j] * lin_stride;
          lin_apply(lo, lin + off, lin_accum + off, lo.z + off, w1[j], n1[j], z1[j], g1[j]);
        }
      }
    }
  }
  if (lane == 0 && leaders && n_unique) atomicAdd(n_unique, leaders);
}

// ---- tf.clip_by_norm per column on the owner (dir_shard_owner_sqnorms, dir_shard_owner_update_clipped)
// A column's norm is over its MERGED per-row sums, and only the owner of a row sees that sum, so every owner reduces
// its own rows per column and the ranks exchange [F][kClipSlices][2] partials:
//   1. per arrival: the leading arrival builds the merged vector exactly as peer_owner_update_kernel does (same
//      leader rule, same __fadd_rn order) and writes its (sum g^2, g1^2) in fp64 to sq[a]; others write zeros.
//      The cost grows with the arrivals, not with the table (no sweep of the slot map).
//   2. CTA (f, s): the column's arrivals of requester q are one contiguous range of q's id segment, found with two
//      lower_bounds: a requester numbers its distinct keys (owner, local row) in sorted order (dir_shard_unique
//      after dir_shard_keys_sort or dir_shard_bag_keys), so each segment is strictly ascending in local row, and a
//      column is a contiguous range of local rows (local row l of rank r is global row l * G + r).  Fixed-order fp64
//      sums, independent of the grid; the partials go to norm[rank] of EVERY rank's norm buffer.
//   3. (after a barrier) peer_clip_combine_kernel: part[f][s] = sum over q of norm[q][f][s] in rank order, so every
//      rank divides by bit-identical denominators.
template <int LPR>
__global__ void __launch_bounds__(256)
peer_owner_sqnorm_kernel(const dir_peer_layout L, const uint32_t* __restrict__ slot,
                         const uint32_t* __restrict__ epoch, int64_t n_local, bool with_g1, double2* __restrict__ sq) {
  constexpr int SLOTS = 32 / LPR;
  constexpr unsigned FULL = 0xffffffffu;
  __shared__ Arrivals s;
  load_arrivals(L, s);
  const uint32_t tag = epoch[0];
  const int64_t total = s.pre[L.G];
  const int G = L.G;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR, grp = lane / LPR;
  const int32_t* ids = reinterpret_cast<const int32_t*>(L.local + L.off_ids);
  const float4* gb = reinterpret_cast<const float4*>(L.local + L.off_g);
  const float* g1b = reinterpret_cast<const float*>(L.local + L.off_g1);
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t a0 = warp * 32; a0 < total; a0 += nwarps * 32) {  // warp-uniform trip count
    const int64_t a = a0 + lane;
    bool lead = false;
    int64_t e = 0, r = 0;
    unsigned long long more = 0;
    if (a < total) {
      const int q = seg_of(s.pre, G, a);
      e = (int64_t)q * L.seg_cap + (a - s.pre[q]);
      r = __ldg(ids + e);
      if (r >= 0 && r < n_local) {
        bool earlier = false;
        for (int p = 0; p < G; ++p) {
          const bool on = (__ldg(slot + r * G + p) >> 24) == tag;
          earlier |= on && p < q;
          if (on && p > q) more |= 1ull << p;
        }
        lead = !earlier;
      }
      if (!lead) sq[a] = make_double2(0.0, 0.0);
    }
    const unsigned lm = __ballot_sync(FULL, lead);
    const int nl = __popc(lm);
    for (int k0 = 0; k0 < nl; k0 += SLOTS) {
      const int n = k0 + grp;
      const bool on = n < nl;
      const int from = on ? (int)__fns(lm, 0, n + 1) : 0;
      const int64_t rr = __shfl_sync(FULL, r, from);
      const int64_t ee = __shfl_sync(FULL, e, from);
      unsigned long long m = __shfl_sync(FULL, more, from);
      double v = 0.0, v1 = 0.0;
      if (on) {
        float4 g = __ldg(gb + ee * LPR + sub);
        float g1 = with_g1 && sub == 0 ? __ldg(g1b + ee) : 0.f;
        while (m) {  // the order of peer_owner_update_kernel: rank
          const int p = __ffsll((long long)m) - 1;
          m &= m - 1;
          const uint32_t sp = __ldg(slot + rr * G + p) & 0xffffffu;
          const int64_t e2 = (int64_t)p * L.seg_cap + (sp - 1u);
          const float4 o = __ldg(gb + e2 * LPR + sub);
          g.x = __fadd_rn(g.x, o.x);
          g.y = __fadd_rn(g.y, o.y);
          g.z = __fadd_rn(g.z, o.z);
          g.w = __fadd_rn(g.w, o.w);
          if (with_g1 && sub == 0) g1 = __fadd_rn(g1, __ldg(g1b + e2));
        }
        v = (double)g.x * g.x + (double)g.y * g.y + (double)g.z * g.z + (double)g.w * g.w;
        v1 = (double)g1 * g1;
      }
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);  // the row's LPR lanes, fixed tree
      if (on && sub == 0) sq[a0 + from] = make_double2(v, v1);
    }
  }
}

// first i < n with a[i] >= x (a ascending)
__device__ __forceinline__ int64_t lower_bound_i32(const int32_t* __restrict__ a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)__ldg(a + mid) < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// grid (F, kClipSlices): slice sl of column f -> norm_peers[every q][rank][f][sl][2]
__global__ void __launch_bounds__(256, 1)
peer_owner_sqnorm_reduce_kernel(const dir_peer_layout L, const double2* __restrict__ sq,
                                const int64_t* __restrict__ local_field_offset, int F,
                                const unsigned long long* __restrict__ norm_peers) {
  __shared__ Arrivals s;
  __shared__ int64_t s_lo[kMaxG], s_hi[kMaxG];
  __shared__ double red[2][256];
  const int f = blockIdx.x, sl = blockIdx.y;
  load_arrivals(L, s);
  const int G = L.G;
  if (threadIdx.x < G) {
    const int q = threadIdx.x;
    const int32_t* seg = reinterpret_cast<const int32_t*>(L.local + L.off_ids) + (int64_t)q * L.seg_cap;
    const int64_t cnt = s.pre[q + 1] - s.pre[q];
    s_lo[q] = lower_bound_i32(seg, cnt, local_field_offset[f]);
    s_hi[q] = lower_bound_i32(seg, cnt, local_field_offset[f + 1]);
  }
  __syncthreads();
  double v = 0.0, v1 = 0.0;
  for (int q = 0; q < G; ++q)
    for (int64_t i = s_lo[q] + (int64_t)sl * 256 + threadIdx.x; i < s_hi[q]; i += (int64_t)kClipSlices * 256) {
      const double2 t = sq[s.pre[q] + i];
      v += t.x;
      v1 += t.y;
    }
  red[0][threadIdx.x] = v;
  red[1][threadIdx.x] = v1;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) {
      red[0][threadIdx.x] += red[0][threadIdx.x + st];
      red[1][threadIdx.x] += red[1][threadIdx.x + st];
    }
    __syncthreads();
  }
  if (threadIdx.x < G) {
    double* dst = reinterpret_cast<double*>(__ldg(norm_peers + threadIdx.x)) +
                  (((int64_t)L.rank * F + f) * kClipSlices + sl) * 2;
    *reinterpret_cast<double2*>(dst) = make_double2(red[0][0], red[1][0]);
  }
}

// part[x] = sum over q of norm[q][x] in rank order, x < F * kClipSlices * 2
__global__ void __launch_bounds__(256)
peer_clip_combine_kernel(const double* __restrict__ norm, int G, int64_t n, double* __restrict__ part) {
  const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= n) return;
  double v = norm[x];
  for (int q = 1; q < G; ++q) v += norm[(int64_t)q * n + x];
  part[x] = v;
}

// ---- TF's Adam on the owner (dir_shard_owner_apply_adam)
// _apply_sparse_shared decays the moments of every row, so the owner sweeps its whole shard in tiles of kAdamTile local
// rows, with adam.cu's tile body.  A tile's gradients come from the requesters' id segments, not from the slot map:
// each segment is strictly ascending in local row (the norm pass relies on it too), so per requester q two warp
// lower_bounds find q's arrivals in [r0, r1), and each arrival i stores (q << 24) | i into the tile's map with an
// integer atomicMin: the lowest requester that asked for a row leads it, the leader rule of peer_owner_update_kernel.
// (2G searches per tile; reading the slot map densely would cost 4G bytes for every row.)  The merged sum starts from
// the leader's and adds the later requesters whose slot cell carries the current epoch, in rank order with __fadd_rn:
// the sum peer_owner_update_kernel applies and peer_owner_sqnorm_kernel squares, bit for bit.
template <int LPR>
struct PeerMergedGrad {
  const float4* gb;    // the exchange buffer's g [G][seg_cap][K]
  const float* g1b;    // and g1 [G][seg_cap]
  const uint32_t* slot;
  int64_t seg_cap;
  uint32_t tag;
  int G;
  bool clipped;
  const int64_t* s_off;
  int F;
  float clip;
  const float* s_den;
  __device__ __forceinline__ float4 load(int key, int sub, int64_t row) const {
    const int q = key >> 24;
    float4 g = __ldg(gb + ((int64_t)q * seg_cap + (key & 0xffffff)) * LPR + sub);
    for (int p = q + 1; p < G; ++p) {
      const uint32_t c = __ldg(slot + row * G + p);
      if ((c >> 24) != tag) continue;
      const float4 o = __ldg(gb + ((int64_t)p * seg_cap + ((c & 0xffffffu) - 1u)) * LPR + sub);
      g.x = __fadd_rn(g.x, o.x);
      g.y = __fadd_rn(g.y, o.y);
      g.z = __fadd_rn(g.z, o.z);
      g.w = __fadd_rn(g.w, o.w);
    }
    return g;
  }
  __device__ __forceinline__ float load_g1(int key, int64_t row) const {
    const int q = key >> 24;
    float g1 = __ldg(g1b + (int64_t)q * seg_cap + (key & 0xffffff));
    for (int p = q + 1; p < G; ++p) {
      const uint32_t c = __ldg(slot + row * G + p);
      if ((c >> 24) == tag) g1 = __fadd_rn(g1, __ldg(g1b + (int64_t)p * seg_cap + ((c & 0xffffffu) - 1u)));
    }
    return g1;
  }
  __device__ __forceinline__ void scale(float4& g, int64_t row) const {
    if (clipped) clip4(g, clip, s_den[field_of(s_off, F, (uint64_t)row)]);
  }
};

template <int LPR>
__global__ void __launch_bounds__(kAdamThreads, 4)
peer_owner_adam_kernel(const dir_peer_layout L, const uint32_t* __restrict__ slot, const uint32_t* __restrict__ epoch,
                       float* table, int64_t row_stride, int64_t n_local, float* lin, float* lin_accum,
                       int64_t lin_stride, const LinOpt lo, const int64_t* __restrict__ field_offset, int F,
                       const double* __restrict__ part, float clip, float lr, float b1, float b2, float eps,
                       const float* __restrict__ beta_power, unsigned long long* n_unique) {
  __shared__ int32_t s_map[kAdamTile];
  __shared__ Arrivals s;
  __shared__ int64_t s_lo[kMaxG], s_hi[kMaxG];
  ClipSmem& cs = clip_smem();
  const bool clipped = part != nullptr;
  if (clipped) clip_denominators(part, field_offset, F, clip, cs.off, cs.den, cs.den1);
  load_arrivals(L, s);                    // (its barrier also publishes the clip factors)
  const AdamStep st = adam_step(lr, b1, b2, eps, beta_power);
  const int G = L.G;
  const int32_t* ids = reinterpret_cast<const int32_t*>(L.local + L.off_ids);
  const PeerMergedGrad<LPR> src{reinterpret_cast<const float4*>(L.local + L.off_g),
                                reinterpret_cast<const float*>(L.local + L.off_g1), slot, L.seg_cap, epoch[0], G,
                                clipped, cs.off, F, clip, cs.den};
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned long long leaders = 0;
  const int64_t n_tiles = (n_local + kAdamTile - 1) / kAdamTile;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * kAdamTile;
    const int64_t r1 = r0 + kAdamTile < n_local ? r0 + kAdamTile : n_local;
    for (int t = warp; t < 2 * G; t += kAdamThreads / 32) {   // requester t / 2: first arrival >= r0 (t even), >= r1
      const int q = t >> 1;
      const int64_t b = warp_lower_bound(reinterpret_cast<const uint32_t*>(ids + (int64_t)q * L.seg_cap),
                                         s.pre[q + 1] - s.pre[q], (uint64_t)((t & 1) ? r1 : r0));
      if (lane == 0) ((t & 1) ? s_hi : s_lo)[q] = b;
    }
    for (int i = threadIdx.x; i < kAdamTile; i += blockDim.x) s_map[i] = -1;
    __syncthreads();
    for (int q = 0; q < G; ++q) {
      const int32_t* seg = ids + (int64_t)q * L.seg_cap;
      for (int64_t i = s_lo[q] + threadIdx.x; i < s_hi[q]; i += blockDim.x)
        atomicMin(reinterpret_cast<unsigned*>(s_map) + (__ldg(seg + i) - r0), ((unsigned)q << 24) | (unsigned)i);
    }
    __syncthreads();
    adam_tile<LPR>(table, row_stride, r0, r1, s_map, st, src);
    for (int i = threadIdx.x; i < (int)(r1 - r0); i += blockDim.x) {
      const int key = s_map[i];
      if (key < 0) continue;
      ++leaders;
      if (lin != nullptr) {               // first-order weights: the leader's merged g1 through the linear rule
        const int64_t row = r0 + i;
        float g1 = src.load_g1(key, row);
        if (clipped) g1 = clip1(g1, clip, cs.den1[field_of(cs.off, F, (uint64_t)row)]);
        const int64_t off = row * lin_stride;
        float n1, z1;
        lin_load(lo, lin_accum, off, n1, z1);
        lin_apply(lo, lin + off, lin_accum + off, lo.z + off, lin[off], n1, z1, g1);
      }
    }
    __syncthreads();                      // s_map / s_lo / s_hi are rewritten by the next tile
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) leaders += __shfl_xor_sync(0xffffffffu, leaders, o);
  if (lane == 0 && leaders && n_unique) atomicAdd(n_unique, leaders);
}

// replicated one-row fields: the G ranks' sums added in rank order, the same update applied to every replica;
// shard_row[j] >= 0 names the row of the sharded table to mirror into (on the rank that owns it)
struct DenseApplyArgs {
  float* table;  // replica: [n_dense] rows, row_stride apart (row | accumulator when Adagrad)
  float* accum;
  int64_t row_stride;
  float* lin;
  float* lin_accum;
  LinOpt lo;  // lo.z: [n_dense]
  RowRule rr;
  float* s_table;  // the sharded table's copy of the row
  float* s_accum;
  int64_t s_row_stride;
  float* s_lin;
  float* s_lin_accum;
  float* s_lin_z;
  int64_t s_lin_stride;
  const int64_t* shard_row;
  unsigned long long* n_unique;
};

// CLIP: a one-row field is a column with one row, so tf.clip_by_norm divides by max(||g||, clip) of the rank-ordered
// sum itself (and the linear weight by max(|g1|, clip)), the arithmetic of dir_embed_bwd_onerow_update(..., clip_norm).
// Every rank forms the same sum: no exchange.
template <int LPR, bool CLIP = false>
__global__ void __launch_bounds__(128)
peer_dense_apply_kernel(const dir_peer_layout L, const char* local_b, const DenseApplyArgs a, float clip = 0.f) {
  constexpr int K = LPR * 4;
  const int j = blockIdx.x, c = threadIdx.x;
  if (!CLIP && c > K) return;
  const int cc = c <= K ? c : K;  // (CLIP keeps every thread until the norm is known)
  float g = 0.f, touched = 0.f;
  for (int b = 0; b < (local_b ? 2 : 1); ++b) {  // buffer (micro-batch), then rank: the same sum on every rank
    const float* gbuf = reinterpret_cast<const float*>((b ? local_b : L.local) + L.off_dense);
    for (int q = 0; q < L.G; ++q) {
      const float* src = gbuf + ((int64_t)q * L.n_dense + j) * (K + 4);
      g = (b == 0 && q == 0) ? src[cc] : __fadd_rn(g, src[cc]);
      touched += src[K + 1];
    }
  }
  if (touched == 0.f) return;  // no rank had a surviving lookup: the row is not touched (the same for every thread)
  if constexpr (CLIP) {
    __shared__ float s_g[K + 1], s_den[2];
    if (c <= K) s_g[c] = g;
    __syncthreads();
    if (c == 0) {
      double sq = 0.0;
      for (int k = 0; k < K; ++k) sq += (double)s_g[k] * s_g[k];
      s_den[0] = fmaxf((float)sqrt(sq), clip);
      s_den[1] = fmaxf(fabsf(s_g[K]), clip);
    }
    __syncthreads();
    if (c > K) return;
    g = clip1(g, clip, s_den[c < K ? 0 : 1]);
  }
  const int64_t sr = __ldg(a.shard_row + j);
  const bool adagrad = a.rr.opt != DIR_OPT_SGD;
  if (c < K) {
    float* tp = a.table + (int64_t)j * a.row_stride + c;
    float acc = 0.f;
    if (adagrad) acc = a.accum[(int64_t)j * a.row_stride + c];
    const float t = upd_rule(*tp, g, acc, a.rr);
    *tp = t;
    if (adagrad) a.accum[(int64_t)j * a.row_stride + c] = acc;
    if (sr >= 0) {
      a.s_table[sr * a.s_row_stride + c] = t;
      if (adagrad) a.s_accum[sr * a.s_row_stride + c] = acc;
    }
  } else {
    if (a.lin != nullptr) {
      float n1, z1;
      lin_load(a.lo, a.lin_accum, j, n1, z1);
      lin_apply(a.lo, a.lin + j, a.lin_accum + j, a.lo.z + j, a.lin[j], n1, z1, g);
      if (sr >= 0) {
        a.s_lin[sr * a.s_lin_stride] = a.lin[j];
        if (a.lo.opt != DIR_OPT_SGD) a.s_lin_accum[sr * a.s_lin_stride] = a.lin_accum[j];
        if (a.lo.opt == DIR_OPT_FTRL) a.s_lin_z[sr * a.s_lin_stride] = a.lo.z[j];
      }
    }
    if (a.n_unique) atomicAdd(a.n_unique, 1ull);
  }
}

// inv[b, f] of the replicated one-row fields: their rows sit behind the exchanged ones (u_cap + j); an id other
// than 0 or a value <= 0 prunes the lookup ([TF] _safe_embedding_lookup_sparse)
__global__ void __launch_bounds__(256)
dense_inv_kernel(const int64_t* __restrict__ idx, const float* __restrict__ val,
                 const int32_t* __restrict__ fields, int n_fields, int64_t B, int F, int64_t tail,
                 int64_t* __restrict__ inv, int* oob_flag) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * n_fields) return;
  const int64_t b = t / n_fields;
  const int j = (int)(t % n_fields);
  const int64_t p = b * F + __ldg(fields + j);
  const int64_t id = __ldg(idx + p);
  const float v = val ? __ldg(val + p) : 1.f;
  if (id > 0 && v > 0.f && oob_flag) *oob_flag = 1;
  inv[p] = (id == 0 && v > 0.f) ? tail + j : -1;
}

static int check_layout(const char* what, const dir_peer_layout* L) {
  if (!L) return fail(DIR_EINVAL, "%s: layout is required", what);
  if (L->G <= 0 || L->G > kMaxG || L->rank < 0 || L->rank >= L->G)
    return fail(DIR_EINVAL, "%s: need 0 <= rank < G <= 64", what);
  if (L->K != 4 && L->K != 8 && L->K != 16 && L->K != 32 && L->K != 64)
    return fail(DIR_EINVAL, "%s: K must be one of 4, 8, 16, 32, 64", what);
  if (L->seg_cap <= 0 || L->u_cap <= 0 || L->n_dense < 0 || L->n_dense > 64)
    return fail(DIR_EINVAL, "%s: seg_cap, u_cap > 0 and 0 <= n_dense <= 64 required", what);
  if (!L->peer_base || !L->local) return fail(DIR_EINVAL, "%s: peer_base and local are required", what);
  if ((reinterpret_cast<uintptr_t>(L->local) & 255u) != 0)
    return fail(DIR_EINVAL, "%s: the exchange buffer must be 256-byte aligned", what);
  return 0;
}

}  // namespace dir

extern "C" int dir_peer_layout_init(int G, int rank, int K, int n_dense, int64_t seg_cap, int64_t u_cap,
                                    dir_peer_layout* out) {
  using namespace dir;
  if (!out) return fail(DIR_EINVAL, "peer_layout_init: out is required");
  if (G <= 0 || G > kMaxG || rank < 0 || rank >= G) return fail(DIR_EINVAL, "peer_layout_init: need 0 <= rank < G <= 64");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "peer_layout_init: K must be one of 4, 8, 16, 32, 64");
  if (seg_cap <= 0 || u_cap <= 0 || n_dense < 0 || n_dense > 64)
    return fail(DIR_EINVAL, "peer_layout_init: seg_cap, u_cap > 0 and 0 <= n_dense <= 64 required");
  out->G = G;
  out->rank = rank;
  out->K = K;
  out->n_dense = n_dense;
  out->seg_cap = seg_cap;
  out->u_cap = u_cap;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off += align_up(bytes, 256);
    return (int64_t)at;
  };
  out->off_hdr = take((size_t)G * 4 * 8);
  out->off_ids = take((size_t)G * seg_cap * 4);
  out->off_rows = take((size_t)(u_cap + n_dense) * K * 4);
  out->off_w = take((size_t)(u_cap + n_dense) * 4);
  out->off_g = take((size_t)G * seg_cap * K * 4);
  out->off_g1 = take((size_t)G * seg_cap * 4);
  out->off_dense = take((size_t)G * (n_dense > 0 ? n_dense : 1) * (K + 4) * 4);
  out->total_bytes = (int64_t)off;
  out->peer_base = nullptr;
  out->local = nullptr;
  return 0;
}

extern "C" int dir_shard_dense_inv(const int64_t* feature_index, const float* feature_value,
                                   const int32_t* onerow_fields, int n_onerow, int64_t B, int F, int64_t tail_row,
                                   int64_t* inv, int* oob_flag, dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0 || n_onerow < 0 || n_onerow > F) return fail(DIR_EINVAL, "shard_dense_inv: bad sizes");
  if (B == 0 || n_onerow == 0) return 0;
  if (!feature_index || !onerow_fields || !inv) return fail(DIR_EINVAL, "shard_dense_inv: null pointer");
  const int64_t n = B * n_onerow;
  dense_inv_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      feature_index, feature_value, onerow_fields, n_onerow, B, F, tail_row, inv, oob_flag);
  return launched("shard_dense_inv");
}

extern "C" int dir_shard_ids_push(const dir_peer_layout* layout, const int32_t* unique_local_rows,
                                  const int64_t* owner_off, int64_t n_capacity, int* err_flag,
                                  uint32_t* slot_epoch, dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_ids_push", layout)) return rc;
  if (!owner_off || !err_flag || n_capacity < 0 || (n_capacity > 0 && !unique_local_rows))
    return fail(DIR_EINVAL, "shard_ids_push: owner_off, err_flag and the id list are required");
  const int64_t want = (n_capacity + 255) / 256;
  const unsigned grid = (unsigned)(want < 1 ? 1 : (want < kPeerCtas ? want : kPeerCtas));
  peer_ids_push_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*layout, unique_local_rows, owner_off,
                                                                           n_capacity, err_flag, slot_epoch);
  return launched("shard_ids_push");
}

extern "C" int dir_shard_slots(const dir_peer_layout* layout, uint32_t* slot, int64_t n_local_rows,
                               const uint32_t* slot_epoch, int* err_flag, int64_t* zero_counter, dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_slots", layout)) return rc;
  if (!slot || !err_flag || !slot_epoch || n_local_rows <= 0)
    return fail(DIR_EINVAL, "shard_slots: slot, slot_epoch, err_flag, n_local_rows > 0 required");
  if (layout->seg_cap >= (1 << 24)) return fail(DIR_EINVAL, "shard_slots: seg_cap must be < 2^24");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  peer_slots_reset_kernel<<<kPeerCtas, 256, 0, st>>>(slot, n_local_rows * layout->G, slot_epoch);
  peer_slots_kernel<<<kPeerCtas, 256, 0, st>>>(*layout, slot, n_local_rows, err_flag, zero_counter, slot_epoch);
  return launched("shard_slots", 2);
}

extern "C" int dir_shard_gather_send(const dir_peer_layout* layout, const float* table, int64_t row_stride,
                                     const float* lin, int64_t lin_stride, const float* dense_table,
                                     int64_t dense_row_stride, const float* dense_lin, int ctas_per_sm,
                                     dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_gather_send", layout)) return rc;
  const int K = layout->K;
  if (!table || row_stride < K || (row_stride & 3) || !aligned16(table))
    return fail(DIR_EINVAL, "shard_gather_send: table (16-byte aligned), row_stride >= K and a multiple of 4 required");
  if (layout->n_dense > 0 && (!dense_table || dense_row_stride < K))
    return fail(DIR_EINVAL, "shard_gather_send: the replicated rows are required when n_dense > 0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned gs_grid = (unsigned)(kSMs * (ctas_per_sm >= 1 && ctas_per_sm <= 8 ? ctas_per_sm : 8));
#define DIR_GS(LP) \
  peer_gather_send_kernel<LP><<<gs_grid, 256, 0, st>>>(*layout, table, row_stride, lin, lin_stride, dense_table, \
                                                       dense_row_stride, dense_lin)
  switch (K / 4) {
    case 1: DIR_GS(1); break;
    case 2: DIR_GS(2); break;
    case 4: DIR_GS(4); break;
    case 8: DIR_GS(8); break;
    default: DIR_GS(16); break;
  }
#undef DIR_GS
  return launched("shard_gather_send");
}

extern "C" int dir_shard_g1_push(const dir_peer_layout* layout, const float* g1_local, const int64_t* owner_off,
                                 int64_t n_capacity, dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_g1_push", layout)) return rc;
  if (!owner_off || n_capacity < 0 || (n_capacity > 0 && !g1_local))
    return fail(DIR_EINVAL, "shard_g1_push: owner_off and g1_local are required");
  const int64_t want = (n_capacity + 255) / 256;
  const unsigned grid = (unsigned)(want < 1 ? 1 : (want < kPeerCtas ? want : kPeerCtas));
  peer_g1_push_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*layout, g1_local, owner_off, n_capacity);
  return launched("shard_g1_push");
}

namespace dir {

// dir_shard_owner_update[_clipped]: clip == nullptr -> the unclipped kernels
static int owner_update(const char* what, const dir_peer_layout* layout, const uint32_t* slot, float* table,
                        float* accum, int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
                        int64_t n_local_rows, const uint32_t* slot_epoch, int optimizer, float lr,
                        const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                        const dir_peer_layout* layout_b, const uint32_t* slot_b, const uint32_t* slot_epoch_b,
                        int64_t* n_unique_out, const OwnerClip* clip, cudaStream_t st) {
  if (int rc = check_layout(what, layout)) return rc;
  if (layout_b != nullptr) {
    if (int rc = check_layout(what, layout_b)) return rc;
    if (!slot_b || !slot_epoch_b || layout_b->G != layout->G || layout_b->seg_cap != layout->seg_cap ||
        layout_b->off_g != layout->off_g || layout->G > 32)
      return fail(DIR_EINVAL, "%s: the second buffer needs its slot map and epoch, the same layout, G <= 32", what);
  }
  const int K = layout->K;
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD && optimizer != DIR_OPT_PROXIMAL_ADAGRAD)
    return fail(DIR_EINVAL, "%s: unknown optimizer", what);
  const RowRule rr{optimizer, lr, table_opt ? table_opt->l1 : 0.f, table_opt ? table_opt->l2 : 0.f};
  if (rr.l1 < 0.f || rr.l2 < 0.f) return fail(DIR_EINVAL, "%s: l1, l2 must be >= 0", what);
  if (!slot || !slot_epoch || !table || n_local_rows <= 0)
    return fail(DIR_EINVAL, "%s: slot, slot_epoch, table, n_local_rows > 0 required", what);
  if (optimizer != DIR_OPT_SGD && !accum) return fail(DIR_EINVAL, "%s: Adagrad needs accum", what);
  if (row_stride < K || (row_stride & 3) || !aligned16(table) || !aligned16(accum))
    return fail(DIR_EINVAL, "%s: rows must be 16-byte aligned, row_stride >= K and a multiple of 4", what);
  LinOpt lo;
  if (int rc = resolve_lin(what, linear_opt, optimizer, lr, lin, lin_accum, lo)) return rc;
  unsigned long long* nu = reinterpret_cast<unsigned long long*>(n_unique_out);  // += (zeroed by dir_shard_slots)
  OwnerSrc src{{layout->local, layout_b ? layout_b->local : nullptr}, {slot, slot_b}, {slot_epoch, slot_epoch_b}};
  const OwnerClip oc = clip ? *clip : OwnerClip{nullptr, nullptr, 0, 0.f};
#define DIR_OU(LP)                                                                                                  \
  if (clip)                                                                                                         \
    peer_owner_update_kernel<LP, 1, true><<<kPeerCtas, 256, 0, st>>>(*layout, src, table, accum, row_stride, lin, \
                                                                        lin_accum, lin_stride, lo, rr, n_local_rows, \
                                                                        nu, oc);                                    \
  else if (layout_b)                                                                                                \
    peer_owner_update_kernel<LP, 2><<<kPeerCtas, 256, 0, st>>>(*layout, src, table, accum, row_stride, lin, lin_accum, \
                                                               lin_stride, lo, rr, n_local_rows, nu, oc);            \
  else                                                                                                              \
    peer_owner_update_kernel<LP, 1><<<kPeerCtas, 256, 0, st>>>(*layout, src, table, accum, row_stride, lin, lin_accum, \
                                                               lin_stride, lo, rr, n_local_rows, nu, oc)
  switch (K / 4) {
    case 1: DIR_OU(1); break;
    case 2: DIR_OU(2); break;
    case 4: DIR_OU(4); break;
    case 8: DIR_OU(8); break;
    default: DIR_OU(16); break;
  }
#undef DIR_OU
  return launched(what);
}

// dir_shard_dense_apply[_clipped]: clip_norm == 0 -> unclipped
static int dense_apply(const char* what, const dir_peer_layout* layout, float* dense_table, float* dense_accum,
                       int64_t row_stride, float* dense_lin, float* dense_lin_accum, int optimizer, float lr,
                       const dir_table_opt* table_opt, const dir_linear_opt* linear_opt, float* shard_table,
                       float* shard_accum, int64_t shard_row_stride, float* shard_lin, float* shard_lin_accum,
                       float* shard_lin_z, int64_t shard_lin_stride, const int64_t* shard_row,
                       const dir_peer_layout* layout_b, int64_t* n_unique_inout, float clip_norm, cudaStream_t st) {
  if (int rc = check_layout(what, layout)) return rc;
  if (layout_b != nullptr) {
    if (int rc = check_layout(what, layout_b)) return rc;
    if (layout_b->off_dense != layout->off_dense || layout_b->G != layout->G)
      return fail(DIR_EINVAL, "%s: the second buffer must have the same layout", what);
  }
  const char* local_b = layout_b ? layout_b->local : nullptr;
  if (layout->n_dense == 0) return 0;
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD && optimizer != DIR_OPT_PROXIMAL_ADAGRAD)
    return fail(DIR_EINVAL, "%s: unknown optimizer", what);
  const RowRule rr{optimizer, lr, table_opt ? table_opt->l1 : 0.f, table_opt ? table_opt->l2 : 0.f};
  if (!dense_table || !shard_row || !shard_table) return fail(DIR_EINVAL, "%s: null pointer", what);
  if (optimizer != DIR_OPT_SGD && (!dense_accum || !shard_accum))
    return fail(DIR_EINVAL, "%s: Adagrad needs the accumulators", what);
  LinOpt lo;
  if (int rc = resolve_lin(what, linear_opt, optimizer, lr, dense_lin, dense_lin_accum, lo)) return rc;
  if (dense_lin && (!shard_lin || (lo.opt != DIR_OPT_SGD && !shard_lin_accum) || (lo.opt == DIR_OPT_FTRL && !shard_lin_z)))
    return fail(DIR_EINVAL, "%s: the sharded copies of the linear state are required", what);
  DenseApplyArgs a{dense_table, dense_accum, row_stride, dense_lin, dense_lin_accum, lo, rr,
                   shard_table, shard_accum, shard_row_stride, shard_lin, shard_lin_accum, shard_lin_z,
                   shard_lin_stride, shard_row, reinterpret_cast<unsigned long long*>(n_unique_inout)};
  const int n = layout->n_dense;
#define DIR_DA(LP)                                                                                       \
  if (clip_norm > 0.f)                                                                                   \
    peer_dense_apply_kernel<LP, true><<<n, 128, 0, st>>>(*layout, local_b, a, clip_norm);               \
  else                                                                                                   \
    peer_dense_apply_kernel<LP><<<n, 128, 0, st>>>(*layout, local_b, a)
  switch (layout->K / 4) {
    case 1: DIR_DA(1); break;
    case 2: DIR_DA(2); break;
    case 4: DIR_DA(4); break;
    case 8: DIR_DA(8); break;
    default: DIR_DA(16); break;
  }
#undef DIR_DA
  return launched(what);
}

}  // namespace dir

extern "C" int dir_shard_owner_update(const dir_peer_layout* layout, const uint32_t* slot, float* table, float* accum,
                                      int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
                                      int64_t n_local_rows, const uint32_t* slot_epoch, int optimizer, float lr,
                                      const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                                      const dir_peer_layout* layout_b,
                                      const uint32_t* slot_b, const uint32_t* slot_epoch_b, int64_t* n_unique_out,
                                      dir_stream_t stream) {
  return dir::owner_update("shard_owner_update", layout, slot, table, accum, row_stride, lin, lin_accum, lin_stride,
                           n_local_rows, slot_epoch, optimizer, lr, table_opt, linear_opt, layout_b, slot_b,
                           slot_epoch_b, n_unique_out, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int dir_shard_dense_apply(const dir_peer_layout* layout, float* dense_table, float* dense_accum,
                                     int64_t row_stride, float* dense_lin, float* dense_lin_accum, int optimizer,
                                     float lr, const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                                     float* shard_table,
                                     float* shard_accum, int64_t shard_row_stride, float* shard_lin,
                                     float* shard_lin_accum, float* shard_lin_z, int64_t shard_lin_stride,
                                     const int64_t* shard_row, const dir_peer_layout* layout_b,
                                     int64_t* n_unique_inout, dir_stream_t stream) {
  return dir::dense_apply("shard_dense_apply", layout, dense_table, dense_accum, row_stride, dense_lin,
                          dense_lin_accum, optimizer, lr, table_opt, linear_opt, shard_table, shard_accum,
                          shard_row_stride, shard_lin, shard_lin_accum, shard_lin_z, shard_lin_stride, shard_row,
                          layout_b, n_unique_inout, 0.f, static_cast<cudaStream_t>(stream));
}

// ---- tf.clip_by_norm per column (see the kernels above)
extern "C" int dir_shard_owner_sqnorms(const dir_peer_layout* layout, const uint32_t* slot, const uint32_t* slot_epoch,
                                       int64_t n_local_rows, const int64_t* local_field_offset, int F, int with_g1,
                                       double* sq_scratch, const uint64_t* norm_peers, dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_owner_sqnorms", layout)) return rc;
  if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "shard_owner_sqnorms: 0 < F <= 1024 required");
  if (!slot || !slot_epoch || !local_field_offset || !sq_scratch || !norm_peers || n_local_rows <= 0)
    return fail(DIR_EINVAL, "shard_owner_sqnorms: slot, slot_epoch, local_field_offset, sq_scratch, norm_peers, "
                            "n_local_rows > 0 required");
  if ((reinterpret_cast<uintptr_t>(sq_scratch) & 15u) != 0)
    return fail(DIR_EINVAL, "shard_owner_sqnorms: sq_scratch must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double2* sq = reinterpret_cast<double2*>(sq_scratch);
  switch (layout->K / 4) {
    case 1: peer_owner_sqnorm_kernel<1><<<kPeerCtas, 256, 0, st>>>(*layout, slot, slot_epoch, n_local_rows, with_g1 != 0, sq); break;
    case 2: peer_owner_sqnorm_kernel<2><<<kPeerCtas, 256, 0, st>>>(*layout, slot, slot_epoch, n_local_rows, with_g1 != 0, sq); break;
    case 4: peer_owner_sqnorm_kernel<4><<<kPeerCtas, 256, 0, st>>>(*layout, slot, slot_epoch, n_local_rows, with_g1 != 0, sq); break;
    case 8: peer_owner_sqnorm_kernel<8><<<kPeerCtas, 256, 0, st>>>(*layout, slot, slot_epoch, n_local_rows, with_g1 != 0, sq); break;
    default: peer_owner_sqnorm_kernel<16><<<kPeerCtas, 256, 0, st>>>(*layout, slot, slot_epoch, n_local_rows, with_g1 != 0, sq); break;
  }
  peer_owner_sqnorm_reduce_kernel<<<dim3((unsigned)F, kClipSlices), 256, 0, st>>>(
      *layout, sq, local_field_offset, F, reinterpret_cast<const unsigned long long*>(norm_peers));
  return launched("shard_owner_sqnorms", 2);
}

extern "C" int dir_shard_owner_update_clipped(const dir_peer_layout* layout, const uint32_t* slot, float* table,
                                              float* accum, int64_t row_stride, float* lin, float* lin_accum,
                                              int64_t lin_stride, int64_t n_local_rows, const uint32_t* slot_epoch,
                                              int optimizer, float lr, const dir_linear_opt* linear_opt,
                                              const int64_t* local_field_offset, int F, const double* norm,
                                              double* partials, float clip_norm, int64_t* n_unique_inout,
                                              dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_owner_update_clipped", layout)) return rc;
  if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "shard_owner_update_clipped: 0 < F <= 1024 required");
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD)
    return fail(DIR_EINVAL, "shard_owner_update_clipped: optimizer must be SGD or Adagrad");
  if (!(clip_norm > 0.f)) return fail(DIR_EINVAL, "shard_owner_update_clipped: clip_norm must be > 0");
  if (!local_field_offset || !norm || !partials) return fail(DIR_EINVAL, "shard_owner_update_clipped: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n = (int64_t)F * kClipSlices * 2;
  peer_clip_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(norm, layout->G, n, partials);
  if (int rc = launched("shard_owner_update_clipped")) return rc;
  const OwnerClip oc{local_field_offset, partials, F, clip_norm};
  return owner_update("shard_owner_update_clipped", layout, slot, table, accum, row_stride, lin, lin_accum, lin_stride,
                      n_local_rows, slot_epoch, optimizer, lr, nullptr, linear_opt, nullptr, nullptr, nullptr,
                      n_unique_inout, &oc, st);
}

extern "C" int dir_shard_dense_apply_clipped(const dir_peer_layout* layout, float* dense_table, float* dense_accum,
                                             int64_t row_stride, float* dense_lin, float* dense_lin_accum,
                                             int optimizer, float lr, const dir_linear_opt* linear_opt,
                                             float* shard_table, float* shard_accum, int64_t shard_row_stride,
                                             float* shard_lin, float* shard_lin_accum, float* shard_lin_z,
                                             int64_t shard_lin_stride, const int64_t* shard_row, float clip_norm,
                                             int64_t* n_unique_inout, dir_stream_t stream) {
  using namespace dir;
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD)
    return fail(DIR_EINVAL, "shard_dense_apply_clipped: optimizer must be SGD or Adagrad");
  if (!(clip_norm > 0.f)) return fail(DIR_EINVAL, "shard_dense_apply_clipped: clip_norm must be > 0");
  return dense_apply("shard_dense_apply_clipped", layout, dense_table, dense_accum, row_stride, dense_lin,
                     dense_lin_accum, optimizer, lr, nullptr, linear_opt, shard_table, shard_accum, shard_row_stride,
                     shard_lin, shard_lin_accum, shard_lin_z, shard_lin_stride, shard_row, nullptr, n_unique_inout,
                     clip_norm, static_cast<cudaStream_t>(stream));
}

// ---- TF's Adam on the owner (see peer_owner_adam_kernel)
extern "C" int dir_shard_owner_apply_adam(const dir_peer_layout* layout, const uint32_t* slot, const uint32_t* slot_epoch,
                                          float* table, int64_t row_stride, int64_t n_local_rows, float* lin,
                                          float* lin_accum, int64_t lin_stride, const dir_linear_opt* linear_opt,
                                          const int64_t* local_field_offset, int F, const double* norm,
                                          double* partials, float clip_norm, const dir_adam_opt* adam,
                                          int64_t* n_unique_inout, dir_stream_t stream) {
  using namespace dir;
  if (int rc = check_layout("shard_owner_apply_adam", layout)) return rc;
  const int K = layout->K;
  if (layout->n_dense != 0)
    return fail(DIR_EINVAL, "shard_owner_apply_adam: n_dense must be 0 (under Adam every field goes through the exchange)");
  if (layout->seg_cap >= (1 << 24)) return fail(DIR_EINVAL, "shard_owner_apply_adam: seg_cap must be < 2^24");
  if (!slot || !slot_epoch) return fail(DIR_EINVAL, "shard_owner_apply_adam: slot and slot_epoch are required");
  if (n_local_rows <= 0 || n_local_rows >= 0xffffffffLL)
    return fail(DIR_EINVAL, "shard_owner_apply_adam: 0 < n_local_rows < 2^32 - 1 required");
  if (!table || row_stride < 3 * K || (row_stride & 3) || !aligned16(table))
    return fail(DIR_EINVAL, "shard_owner_apply_adam: rows are [T | m | v]: row_stride >= 3K, a multiple of 4, table "
                            "16-byte aligned");
  if (!adam || !adam->beta_power) return fail(DIR_EINVAL, "shard_owner_apply_adam: adam and its beta_power are required");
  if (!(adam->lr > 0.f)) return fail(DIR_EINVAL, "shard_owner_apply_adam: lr must be > 0");
  if (!(adam->beta1 >= 0.f && adam->beta1 < 1.f) || !(adam->beta2 >= 0.f && adam->beta2 < 1.f))
    return fail(DIR_EINVAL, "shard_owner_apply_adam: 0 <= beta1, beta2 < 1 required");
  if (!(adam->epsilon > 0.f)) return fail(DIR_EINVAL, "shard_owner_apply_adam: epsilon must be > 0");
  if (norm) {
    if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "shard_owner_apply_adam: 0 < F <= 1024 required");
    if (!local_field_offset) return fail(DIR_EINVAL, "shard_owner_apply_adam: the clip needs local_field_offset");
    if (!partials) return fail(DIR_EINVAL, "shard_owner_apply_adam: the clip needs partials");
    if (!(clip_norm > 0.f)) return fail(DIR_EINVAL, "shard_owner_apply_adam: clip_norm must be > 0");
  }
  LinOpt lo{DIR_OPT_SGD, 0.f, 0.f, 0.f, nullptr};
  if (lin != nullptr) {
    if (!linear_opt)
      return fail(DIR_EINVAL, "shard_owner_apply_adam: lin needs linear_opt (Adam does not train first-order weights)");
    if (int rc = resolve_lin("shard_owner_apply_adam", linear_opt, DIR_OPT_SGD, 0.f, lin, lin_accum, lo)) return rc;
    if (lin_stride < 1) return fail(DIR_EINVAL, "shard_owner_apply_adam: lin_stride must be >= 1");
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (norm) {                             // the rank-order combine of dir_shard_owner_update_clipped
    const int64_t n = (int64_t)F * kClipSlices * 2;
    peer_clip_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(norm, layout->G, n, partials);
  }
  const int64_t n_tiles = (n_local_rows + kAdamTile - 1) / kAdamTile;
  const unsigned grid = (unsigned)(n_tiles < (int64_t)kSMs * 4 ? n_tiles : (int64_t)kSMs * 4);
  const double* part = norm ? partials : nullptr;
  unsigned long long* nu = reinterpret_cast<unsigned long long*>(n_unique_inout);
  const float b1 = adam->beta1, b2 = adam->beta2;
#define DIR_OA(LP)                                                                                                  \
  peer_owner_adam_kernel<LP><<<grid, kAdamThreads, 0, st>>>(*layout, slot, slot_epoch, table, row_stride,          \
                                                            n_local_rows, lin, lin_accum, lin_stride, lo,           \
                                                            local_field_offset, F, part, clip_norm, adam->lr, b1,   \
                                                            b2, adam->epsilon, adam->beta_power, nu)
  switch (K / 4) {
    case 1: DIR_OA(1); break;
    case 2: DIR_OA(2); break;
    case 4: DIR_OA(4); break;
    case 8: DIR_OA(8); break;
    default: DIR_OA(16); break;
  }
#undef DIR_OA
  adam_advance_powers(adam->beta_power, b1, b2, st);
  return launched("shard_owner_apply_adam", norm ? 3 : 2);
}
