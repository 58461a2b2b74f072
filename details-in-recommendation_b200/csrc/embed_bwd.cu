// K6+K7: deterministic backward of lookup + first order + FM with the sparse row-wise
// Adagrad / SGD update fused in.
//
//   sort      (global row, lookup position) pairs, stable LSD radix sort
//   phase 1   the sorted list is cut into fixed chunks of C lookups; LPR = K/4 lanes walk one
//             chunk in order, forming each lookup's gradient on the fly from g[b], S[b,:], u[b,f,:]
//             and the row (the [B*F,K] per-lookup gradient is never materialised) and summing runs
//             of equal rows sequentially (= sample order, the order TF's CPU UnsortedSegmentSum
//             uses).  A run that lies inside its chunk is final: its row is updated right there.
//             A run that crosses a chunk boundary leaves a partial sum in the workspace.
//   phase 2   the chunk where a crossing run starts adds the partials of the following chunks in
//             chunk order and updates the row; runs longer than kLongRun chunks go to
//   phase 3   one CTA per long run: strided sequential sums + a fixed-shape tree.
// Chunking depends only on positions in the sorted list, so the result is bit-identical from
// run to run; there are no floating-point atomics.
//
// Reference: TF autodiff + optimizer.minimize behind models/DeepFM/deepFM.py:230-241
// (SURVEY.md rows A8/A9).
#include <type_traits>

#include "common.cuh"
#include "keys.cuh"
#include "radix.cuh"
#include "update.cuh"

namespace dir {

constexpr int kTile = 32;     // lookups a warp handles at a time
constexpr int kChunk = 128;   // lookups per chunk (C): one warp walks one chunk
constexpr int kLongRun = 32;  // chunks; longer crossing runs go to phase 3
constexpr uint32_t kNoKey = 0xffffffffu;
constexpr int kOneRowCtasMax = 444;  // CTAs of the one-row column-sum kernel (three per SM)

struct BwdWorkspace {
  uint32_t* keys;      // [n] sorted global rows
  uint32_t* pos;       // [n] lookup position b*F+f of each sorted entry
  uint32_t* pos_in;    // [n] the other half of the radix sort's ping-pong for the values
  uint32_t* alt_keys;  // [n] the other half of the radix sort's ping-pong for the keys
  uint32_t* radix_hist; // radix_hist_bytes(n)
  float* part;         // [nchunks][2][K]
  float* part1;        // [nchunks][2]
  uint32_t* long_list; // [nchunks / kLongRun + 1]
  uint32_t* long_count;
  unsigned long long* n_unique;
  int* onerow_flags;   // [64]
  double* onerow_part; // [296][64][K + 4] fp64 partial column sums
  size_t total;
};

static BwdWorkspace carve(void* base, int64_t n, int K) {
  BwdWorkspace w;
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* r = p ? p + off : nullptr;
    off += align_up(bytes, 256);
    return r;
  };
  const int64_t nchunks = (n + kChunk - 1) / kChunk;
  w.keys = reinterpret_cast<uint32_t*>(take((size_t)n * 4));
  w.pos = reinterpret_cast<uint32_t*>(take((size_t)n * 4));
  w.pos_in = reinterpret_cast<uint32_t*>(take((size_t)n * 4));
  w.alt_keys = reinterpret_cast<uint32_t*>(take((size_t)n * 4));
  w.radix_hist = reinterpret_cast<uint32_t*>(take(radix_hist_bytes(n)));
  // everything whose size does not depend on K comes first: the sort step carves with a dummy K
  w.long_list = reinterpret_cast<uint32_t*>(take((size_t)(nchunks / kLongRun + 1) * 4));
  w.long_count = reinterpret_cast<uint32_t*>(take(16));
  w.n_unique = reinterpret_cast<unsigned long long*>(w.long_count ? (char*)w.long_count + 8 : nullptr);
  w.onerow_flags = reinterpret_cast<int*>(take(64 * 4));
  w.part1 = reinterpret_cast<float*>(take((size_t)nchunks * 2 * 4));
  w.part = reinterpret_cast<float*>(take((size_t)nchunks * 2 * K * 4));
  w.onerow_part = reinterpret_cast<double*>(take((size_t)kOneRowCtasMax * 64 * (K + 4) * 8));
  w.total = off;
  return w;
}

// Every field has a default, so each entry point names only the fields of its own mode.
struct BwdArgs {
  float* table = nullptr;
  float* accum = nullptr;
  int64_t row_stride = 0;
  float* lin = nullptr;
  float* lin_accum = nullptr;
  int64_t lin_stride = 0;
  const float* val = nullptr;
  const float* g_first = nullptr;
  const float* g_fm = nullptr;
  const float* S = nullptr;
  const float* u = nullptr;
  const uint32_t* keys = nullptr;
  const uint32_t* pos = nullptr;
  float* part = nullptr;
  float* part1 = nullptr;
  uint32_t* long_list = nullptr;
  uint32_t* long_count = nullptr;
  unsigned long long* n_unique = nullptr;
  int64_t n = 0;
  int F = 0;
  uint32_t pruned_key = 0;  // = n_rows
  int opt = DIR_OPT_SGD;
  float lr = 0.f;
  uint32_t div_magic = 0;   // position / F == (position * div_magic) >> div_shift for position < 2^31
  int div_shift = 0;
  const int32_t* field_sel = nullptr;  // sorted entries index the compact [B, n_sel] list of these fields (or NULL)
  int n_sel = 0;
  // sharded-table modes (see kMode*)
  int mode = 0;
  const uint32_t* rowidx = nullptr;  // kModeEmit: row of `table` (the exchanged unique-row buffer) per sorted entry
  float* emit = nullptr;             // kModeEmit: [n_unique, emit_stride] receives (G[K], g1) per run
  int64_t emit_stride = 0;
  // kModeEmit straight into the owners' buffers over NVLink (emit_peers != NULL; csrc/shard_peer.cu): distinct
  // row u of segment q (emit_seg[q] <= u < emit_seg[q+1]) is row emit_dst_row + u - emit_seg[q] of the gradient
  // region (emit_byte_off) of the buffer at the peer-mapped address emit_peers[q]; its g1 goes to emit_g1[u]
  const int64_t* emit_seg = nullptr;
  const int64_t* emit_peers = nullptr;
  int64_t emit_byte_off = 0;
  int64_t emit_dst_row = 0;
  int64_t emit_seg_cap = 0;
  float* emit_g1 = nullptr;
  int emit_G = 0;
  int perm_G = 0, perm_rank = 0;  // > 1: warps take the chunks in an owner-interleaved, rank-rotated order (see chunk_of)
  int64_t perm_M = 0;
  int emit_read_key = 0;  // kModeEmit over the table itself: rows are read at the key, sums still go to row uidx of `emit`
  LinOpt lo{};
  // kModeBag (multi-hot bags, embed_bag.cu): sorted payload = entry index j
  const uint32_t* entry_slot = nullptr;  // [nnz] slot b*F+f of entry j
  const float* entry_x = nullptr;        // [nnz] effective scale w_j / norm(bag)
  const float* emb = nullptr;            // [B*F, K] combined embeddings e_s saved by the forward
  float l1 = 0.f, l2 = 0.f;              // ProximalAdagrad strengths of the table rows
};

// one distinct row's sums: LPR lanes store the K-vector; g1 follows it in a local emit row, or goes to emit_g1[u]
// when the rows cross NVLink (64-byte rows there: whole 16-byte stores only, g1 is shipped in bulk afterwards)
template <int LPR>
__device__ __forceinline__ void emit_store(const BwdArgs& a, uint32_t u, int sub, float4 G, float g1) {
  if (a.emit_peers == nullptr) {
    float* e = a.emit + (int64_t)u * a.emit_stride;
    *(reinterpret_cast<float4*>(e) + sub) = G;
    if (sub == 0) e[LPR * 4] = g1;
    return;
  }
  int q = 0;
  for (int g = 1; g < a.emit_G; ++g) q += ((int64_t)u >= __ldg(a.emit_seg + g)) ? 1 : 0;
  const int64_t j = (int64_t)u - __ldg(a.emit_seg + q);
  if (j < a.emit_seg_cap) {  // (the id push flagged the overflow; never store out of bounds)
    float4* base = reinterpret_cast<float4*>(__ldg(a.emit_peers + q) + a.emit_byte_off);
    base[(a.emit_dst_row + j) * LPR + sub] = G;
  }
  if (sub == 0) a.emit_g1[u] = g1;
}

constexpr int kModeLocal = 0;  // gradients formed from g, S, u, row; the row is updated in place
constexpr int kModeEmit = 1;   // requester side of a sharded table: per-row sums go to `emit`
constexpr int kModeBag = 3;    // multi-hot bags: entry j of slot s contributes x_j (g_fm (S - e_s) + u_s)
constexpr int kModeBagEmit = 4;  // requester side of a sharded table fed with bags: kModeBag's gradients, kModeEmit's sums
__host__ __device__ constexpr bool mode_emits(int m) { return m == kModeEmit || m == kModeBagEmit; }
__host__ __device__ constexpr bool mode_bags(int m) { return m == kModeBag || m == kModeBagEmit; }

template <int LPR>
__device__ __forceinline__ void apply_update(const BwdArgs& a, uint32_t key, int sub, float4 G,
                                             float g1) {
  if (mode_emits(a.mode)) {  // `key` is the row of the emit buffer here
    emit_store<LPR>(a, key, sub, G, g1);
    return;
  }
  const bool adagrad = a.opt != DIR_OPT_SGD;  // the rule keeps an accumulator
  const RowRule rr{a.opt, a.lr, a.l1, a.l2};
  float4* trow = reinterpret_cast<float4*>(a.table + (int64_t)key * a.row_stride) + sub;
  float4 T = *trow;
  float4 A = make_float4(0.f, 0.f, 0.f, 0.f);
  float4* arow = nullptr;
  if (adagrad) {
    arow = reinterpret_cast<float4*>(a.accum + (int64_t)key * a.row_stride) + sub;
    A = *arow;
  }
  T.x = upd_rule(T.x, G.x, A.x, rr);
  T.y = upd_rule(T.y, G.y, A.y, rr);
  T.z = upd_rule(T.z, G.z, A.z, rr);
  T.w = upd_rule(T.w, G.w, A.w, rr);
  *trow = T;
  if (adagrad) *arow = A;
  if (a.lin != nullptr && sub == 0) {
    const int64_t off = (int64_t)key * a.lin_stride;
    float n1, z1;
    lin_load(a.lo, a.lin_accum, off, n1, z1);
    lin_apply(a.lo, a.lin + off, a.lin_accum + off, a.lo.z + off, a.lin[off], n1, z1, g1);
  }
}

// Row update from values already in registers (same arithmetic as apply_update).
__device__ __forceinline__ void apply_loaded(const BwdArgs& a, uint32_t key, int sub, float4 T,
                                             float4 A, float4 G, float w, float a1, float z1, float g1) {
  const bool adagrad = a.opt != DIR_OPT_SGD;
  const RowRule rr{a.opt, a.lr, a.l1, a.l2};
  T.x = upd_rule(T.x, G.x, A.x, rr);
  T.y = upd_rule(T.y, G.y, A.y, rr);
  T.z = upd_rule(T.z, G.z, A.z, rr);
  T.w = upd_rule(T.w, G.w, A.w, rr);
  *(reinterpret_cast<float4*>(a.table + (int64_t)key * a.row_stride) + sub) = T;
  if (adagrad) *(reinterpret_cast<float4*>(a.accum + (int64_t)key * a.row_stride) + sub) = A;
  if (a.lin != nullptr && sub == 0) {
    const int64_t off = (int64_t)key * a.lin_stride;
    lin_apply(a.lo, a.lin + off, a.lin_accum + off, a.lo.z + off, w, a1, z1, g1);
  }
}

// phase 1: one warp per chunk of kChunk sorted lookups, kTile = 32 at a time.
//   lane-per-lookup stage : key, position, sample = position / F, value, g_first, g_fm
//   vector stage          : LPR lanes hold one K-vector as float4s, so a pass covers 32/LPR lookups;
//                           PB passes have their S / u / row loads in flight together.  Each pass forms
//                           the per-lookup gradients, sums runs of equal rows with a segmented
//                           inclusive scan over the row slots (fixed shuffle pattern) and adds the
//                           running sum carried from the previous pass.
//   At the last lookup of a run: the run lies inside the chunk -> update the row right here with the
//   row / accumulator already in registers; otherwise leave a partial for phase 2 / 3.
template <int LPR, int MODE>
__global__ void __launch_bounds__(256, 3) embed_bwd_reduce_kernel(const BwdArgs a) {
  constexpr int K = LPR * 4;
  constexpr int SLOTS = 32 / LPR;             // lookups per pass
  constexpr int PASSES = LPR;                 // passes per tile of 32 lookups
  constexpr int PB = PASSES < 2 ? PASSES : 2; // passes whose loads are in flight together
  constexpr unsigned FULL = 0xffffffffu;
  constexpr bool EMIT = mode_emits(MODE), BAG = mode_bags(MODE);
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR;
  const int slot = lane / LPR;
  // Which chunk this warp walks.  When the sums go straight to their owners over NVLink, the sorted list is
  // owner-major: in chunk order every rank would write to owner 0 first, then owner 1, ... and that owner's NVLink
  // ingress would serve all ranks at once.  Virtual chunk v -> chunk ((v + rank) mod G) * M + v / G (M = chunks / G
  // rounded up) interleaves the owners and starts every rank on a different one.  The chunking itself -- and with it
  // every sum -- is unchanged.
  int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (a.perm_G > 1) chunk = (int64_t)((chunk + a.perm_rank) % a.perm_G) * a.perm_M + chunk / a.perm_G;
  const int64_t i0 = chunk * kChunk;
  const int64_t n = a.n;
  if (i0 >= n) return;  // whole warp
  const int64_t chunk_end = min(n, i0 + (int64_t)kChunk);
  const uint32_t prev_key = i0 > 0 ? __ldg(a.keys + i0 - 1) : kNoKey;
  const uint32_t next_chunk_key = chunk_end < n ? __ldg(a.keys + chunk_end) : kNoKey;
  const bool adagrad = a.opt != DIR_OPT_SGD;
  // L2 policies.  A 64-byte gradient / row gather pulls a whole 128-byte line from HBM (measured,
  // tools/gather_probe.cu); the other half of a `u` line belongs to the neighbouring field of the
  // same sample and is wanted later by some other warp, so `u` lines are asked to stay (evict_last)
  // while row / accumulator lines, read and rewritten exactly once, are asked to leave first.
  const uint64_t pol_once = policy_evict_last();
  const uint64_t pol_row = policy_evict_first();

  uint32_t carry_key = kNoKey, last_key = prev_key;
  float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
  float carry1 = 0.f;
  unsigned heads = 0;

  // software pipeline: the next tile's keys / positions are requested before this tile's gathers
  int64_t i = i0 + lane;
  uint32_t key_nx = i < chunk_end ? __ldg(a.keys + i) : a.pruned_key;
  uint32_t pos_nx = i < chunk_end ? __ldg(a.pos + i) : 0u;
  uint32_t row_nx = key_nx;  // row of `table` this lookup reads
  if (EMIT) row_nx = i < chunk_end ? __ldg(a.rowidx + i) : 0u;

  for (int64_t base = i0; base < chunk_end; base += kTile) {
    const uint32_t key = key_nx, row = row_nx;
    uint32_t pos = pos_nx;
    i = base + kTile + lane;
    key_nx = i < chunk_end ? __ldg(a.keys + i) : a.pruned_key;
    pos_nx = i < chunk_end ? __ldg(a.pos + i) : 0u;
    row_nx = key_nx;
    if (EMIT) row_nx = i < chunk_end ? __ldg(a.rowidx + i) : 0u;

    // ---- lane-per-lookup stage
    const bool valid = key != a.pruned_key;
    uint32_t keyp = __shfl_up_sync(FULL, key, 1);
    if (lane == 0) keyp = last_key;
    uint32_t keyn = __shfl_down_sync(FULL, key, 1);
    const uint32_t first_nx = __shfl_sync(FULL, key_nx, 0);
    if (lane == 31) keyn = base + kTile < chunk_end ? first_nx : next_chunk_key;
    const bool last_in_chunk = base + lane == chunk_end - 1;
    if (last_in_chunk) keyn = next_chunk_key;
    last_key = __shfl_sync(FULL, key, 31);
    heads += __popc(__ballot_sync(FULL, valid && key != keyp));
    const unsigned cont = __ballot_sync(FULL, valid && keyn == key);  // run goes on after this lookup
    float v = 1.f, g2 = 0.f, d1l = 0.f, wraw = 1.f;
    if (BAG) {  // payload = entry index: fetch its slot, scale and raw weight; pos becomes the slot
      const uint32_t j = pos;
      pos = valid ? __ldg(a.entry_slot + j) : 0u;
      if (valid) {
        v = __ldg(a.entry_x + j);
        if (a.val) wraw = __ldg(a.val + j);
      }
    }
    // sample of this lookup: entry / (fields per sample in the sorted list)
    const uint32_t b = (uint32_t)(((uint64_t)pos * a.div_magic) >> a.div_shift);
    if (a.field_sel != nullptr)  // compact list of selected fields -> position in the [B, F] inputs
      pos = b * (uint32_t)a.F + (uint32_t)__ldg(a.field_sel + (pos - b * (uint32_t)a.n_sel));
    if (valid) {
      if (BAG) {
        if (a.g_first) d1l = __fmul_rn(__ldg(a.g_first + b), wraw);   // first order combines with 'sum'
        g2 = __ldg(a.g_fm + b);
      } else {
        if (a.val) v = __ldg(a.val + pos);
        if (a.g_first) d1l = __ldg(a.g_first + b);
        g2 = __ldg(a.g_fm + b);
        d1l = __fmul_rn(d1l, v);
      }
    }
    // what happens at this lookup: 0 nothing, 1 finish the row (update / emit), 2 partial (run open
    // to the left), 3 partial (run starts here, open to the right); bits 2.. = scan mask: bit t set
    // when the lookup 2^t places earlier in the same pass has the same key
    int act = 0;
    if (valid && (keyn != key || last_in_chunk)) {
      const bool left_open = key == prev_key;
      const bool right_open = last_in_chunk && keyn == key;
      act = (!left_open && !right_open) ? 1 : (left_open ? 2 : 3);
    }
#pragma unroll
    for (int t = 0; (1 << t) < SLOTS; ++t) {
      const uint32_t ko = __shfl_up_sync(FULL, key, 1 << t);
      if ((lane % SLOTS) >= (1 << t) && ko == key && valid) act |= 4 << t;
    }

    // ---- vector stage
#pragma unroll
    for (int j0 = 0; j0 < PASSES; j0 += PB) {
      uint32_t k[PB], rw[PB];
      int ac[PB];
      float a1[PB], lw[PB], lz[PB];
      float4 Sb[PB], ub[PB], T[PB], A[PB];
      float4 Rw[MODE == kModeBag ? PB : 1];  // kModeBag: the row itself (T holds the combined e_s)
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const int l = (j0 + j) * SLOTS + slot;
        k[j] = __shfl_sync(FULL, key, l);
        rw[j] = EMIT ? __shfl_sync(FULL, row, l) : k[j];
        const uint32_t p = __shfl_sync(FULL, pos, l);
        const uint32_t bb = __shfl_sync(FULL, b, l);
        ac[j] = __shfl_sync(FULL, act, l);
        Sb[j] = ub[j] = T[j] = A[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        lw[j] = a1[j] = lz[j] = 0.f;
        if (k[j] != a.pruned_key) {
          const int64_t ro = (int64_t)((EMIT && a.emit_read_key) ? k[j] : rw[j]) * a.row_stride;
          // (S before u: the other order spills 8 bytes at K = 32 and 64.  A 64-byte L2 fill for one field's slice
          // of u measured slower: the neighbouring field's slice is no longer left in L2 for the warp that wants it)
          Sb[j] = __ldg(reinterpret_cast<const float4*>(a.S + (int64_t)bb * K) + sub);
          if (a.u) ub[j] = ldg_hint(a.u + (int64_t)p * K + sub * 4, pol_once);
          if (BAG) {
            T[j] = __ldg(reinterpret_cast<const float4*>(a.emb + (int64_t)p * K) + sub);
          } else {
            // coherent load: this warp may rewrite the row further down
            T[j] = ld_hint(a.table + ro + sub * 4, pol_row);
          }
          if (!EMIT && (ac[j] & 3) == 1) {
            if (MODE == kModeBag) Rw[j] = ld_hint(a.table + ro + sub * 4, pol_row);
            if (adagrad) A[j] = ld_hint(a.accum + ro + sub * 4, pol_row);
            if (a.lin != nullptr && sub == 0) {
              lw[j] = a.lin[(int64_t)rw[j] * a.lin_stride];
              lin_load(a.lo, a.lin_accum, (int64_t)rw[j] * a.lin_stride, a1[j], lz[j]);
            }
          }
        }
      }
#pragma unroll
      for (int j = 0; j < PB; ++j) {
        const int l = (j0 + j) * SLOTS + slot;
        float4 d;
        float d1 = __shfl_sync(FULL, d1l, l);
        // value * (g_fm * (S - value*T) + u), evaluation order of the oracle
        const float x = __shfl_sync(FULL, v, l), gg = __shfl_sync(FULL, g2, l);
        // e of this lookup: value * row, or (bags) the combined embedding of its slot
        const float xe = BAG ? 1.f : x;
        d.x = __fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[j].x, __fmul_rn(xe, T[j].x))), ub[j].x));
        d.y = __fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[j].y, __fmul_rn(xe, T[j].y))), ub[j].y));
        d.z = __fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[j].z, __fmul_rn(xe, T[j].z))), ub[j].z));
        d.w = __fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[j].w, __fmul_rn(xe, T[j].w))), ub[j].w));
        if (k[j] == a.pruned_key) {
          d = make_float4(0.f, 0.f, 0.f, 0.f);
          d1 = 0.f;
        }
        // segmented inclusive scan over the row slots (sorted: equal keys are contiguous); a step is
        // skipped when no lookup of the pass needs it (most runs are short)
#pragma unroll
        for (int t = 0; (1 << t) < SLOTS; ++t) {
          if (__any_sync(FULL, ac[j] & (4 << t))) {
            const int dl = (1 << t) * LPR;
            const float ox = __shfl_up_sync(FULL, d.x, dl);
            const float oy = __shfl_up_sync(FULL, d.y, dl);
            const float oz = __shfl_up_sync(FULL, d.z, dl);
            const float ow = __shfl_up_sync(FULL, d.w, dl);
            const float o1 = __shfl_up_sync(FULL, d1, dl);
            if (ac[j] & (4 << t)) {
              d.x = __fadd_rn(ox, d.x);
              d.y = __fadd_rn(oy, d.y);
              d.z = __fadd_rn(oz, d.z);
              d.w = __fadd_rn(ow, d.w);
              d1 = __fadd_rn(o1, d1);
            }
          }
        }
        if (carry_key != kNoKey && k[j] == carry_key) {  // the run came in from an earlier pass
          d.x = __fadd_rn(carry.x, d.x);
          d.y = __fadd_rn(carry.y, d.y);
          d.z = __fadd_rn(carry.z, d.z);
          d.w = __fadd_rn(carry.w, d.w);
          d1 = __fadd_rn(carry1, d1);
        }
        if ((ac[j] & 3) == 1) {
          if (EMIT) {
            emit_store<LPR>(a, rw[j], sub, d, d1);
          } else {
            apply_loaded(a, rw[j], sub, MODE == kModeBag ? Rw[j] : T[j], A[j], d, lw[j], a1[j], lz[j], d1);
          }
        } else if ((ac[j] & 3) >= 2) {
          const int64_t s = chunk * 2 + ((ac[j] & 3) == 2 ? 0 : 1);
          *(reinterpret_cast<float4*>(a.part + s * K) + sub) = d;
          if (sub == 0) a.part1[s] = d1;
        }
        // hand the running sum to the next pass only when the run really continues (warp-uniform)
        carry_key = kNoKey;
        if ((cont >> ((j0 + j) * SLOTS + SLOTS - 1)) & 1u) {
          const int src = (SLOTS - 1) * LPR + sub;
          carry_key = __shfl_sync(FULL, k[j], src);
          carry.x = __shfl_sync(FULL, d.x, src);
          carry.y = __shfl_sync(FULL, d.y, src);
          carry.z = __shfl_sync(FULL, d.z, src);
          carry.w = __shfl_sync(FULL, d.w, src);
          carry1 = __shfl_sync(FULL, d1, src);
        }
      }
    }
  }
  if (lane == 0 && heads && a.n_unique) atomicAdd(a.n_unique, (unsigned long long)heads);
}

// phase 2 + 3 in one launch.  Phase 2: one lane group per chunk; the chunk where a crossing run
// starts adds the partials of the following chunks in chunk order and finishes the row.  A run that
// spans more than kLongRun chunks is left to phase 3: the whole CTA finds its end by probing chunk
// heads in parallel, sums the partials strided over lane groups (sequential per group) and combines
// the groups with a fixed-shape tree.
// (six CTAs per SM keeps 40 registers; without the bound ptxas took 48)
template <int LPR>
__global__ void __launch_bounds__(256, 6) embed_bwd_finish_kernel(const BwdArgs a, int64_t* n_unique_out) {
  constexpr int K = LPR * 4;
  constexpr int NG = 256 / LPR;  // lane groups per CTA
  __shared__ float4 sm[256];
  __shared__ float sm1[NG];
  __shared__ uint32_t s_long[NG];
  __shared__ int s_nlong;
  if (threadIdx.x == 0) s_nlong = 0;
  __syncthreads();
  const int q = threadIdx.x / LPR;
  const int sub = threadIdx.x % LPR;
  const int64_t n = a.n;
  {
    const int64_t gid = (int64_t)blockIdx.x * NG + q;
    const int64_t i0 = gid * kChunk;
    const int64_t end = min(n, i0 + (int64_t)kChunk);
    bool head = i0 < n && end < n;  // the last chunk cannot be open to the right
    uint32_t key = 0;
    if (head) {
      key = __ldg(a.keys + end - 1);
      head = key != a.pruned_key && __ldg(a.keys + end) == key &&      // open to the right
             !(i0 > 0 && __ldg(a.keys + i0 - 1) == key);               // and not a middle piece
    }
    if (head) {
      const int64_t far = (gid + 1 + kLongRun) * kChunk;  // chunk gid+1+kLongRun still starts with key?
      if (far < n && __ldg(a.keys + far) == key) {
        if (sub == 0) s_long[atomicAdd(&s_nlong, 1)] = (uint32_t)gid;
      } else {
        float4 acc = *(reinterpret_cast<const float4*>(a.part + (gid * 2 + 1) * K) + sub);
        float acc1 = a.part1[gid * 2 + 1];
        for (int64_t j = gid + 1; j * kChunk < n && __ldg(a.keys + j * kChunk) == key; ++j) {
          const float4 p = *(reinterpret_cast<const float4*>(a.part + (j * 2) * K) + sub);
          acc.x = __fadd_rn(acc.x, p.x);
          acc.y = __fadd_rn(acc.y, p.y);
          acc.z = __fadd_rn(acc.z, p.z);
          acc.w = __fadd_rn(acc.w, p.w);
          acc1 = __fadd_rn(acc1, a.part1[j * 2]);
        }
        apply_update<LPR>(a, mode_emits(a.mode) ? __ldg(a.rowidx + end - 1) : key, sub, acc, acc1);
      }
    }
  }
  __syncthreads();
  const int n_long = s_nlong;
  for (int r = 0; r < n_long; ++r) {
    // the order of s_long depends on the atomics, but each run is finished on its own
    const int64_t gid = s_long[r];
    const int64_t first = (gid + 1) * kChunk;
    const uint32_t key = __ldg(a.keys + first - 1);
    int64_t M = 0;  // chunks gid+1 .. gid+M start with `key`: they hold a left-open partial
    for (;;) {
      const int64_t c = gid + 1 + M + threadIdx.x;
      const int ok = c * kChunk < n && __ldg(a.keys + c * kChunk) == key;
      const int cnt = __syncthreads_count(ok);
      M += cnt;
      if (cnt < 256) break;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float acc1 = 0.f;
    for (int64_t m = q; m < M; m += NG) {
      const int64_t j = gid + 1 + m;
      const float4 p = *(reinterpret_cast<const float4*>(a.part + (j * 2) * K) + sub);
      acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
      if (sub == 0) acc1 += a.part1[j * 2];
    }
    sm[threadIdx.x] = acc;
    if (sub == 0) sm1[q] = acc1;
    __syncthreads();
#pragma unroll
    for (int st = NG / 2; st > 0; st >>= 1) {
      if (q < st) {
        const float4 o = sm[threadIdx.x + st * LPR];
        float4 m = sm[threadIdx.x];
        m.x += o.x; m.y += o.y; m.z += o.z; m.w += o.w;
        sm[threadIdx.x] = m;
        if (sub == 0) sm1[q] += sm1[q + st];
      }
      __syncthreads();
    }
    if (q == 0) {
      const float4 h = *(reinterpret_cast<const float4*>(a.part + (gid * 2 + 1) * K) + sub);
      float4 t = sm[threadIdx.x];
      t.x += h.x; t.y += h.y; t.z += h.z; t.w += h.w;
      apply_update<LPR>(a, mode_emits(a.mode) ? __ldg(a.rowidx + first - 1) : key, sub, t,
                        a.part1[gid * 2 + 1] + sm1[0]);
    }
    __syncthreads();
  }
  // every atomicAdd of phase 1 has landed: publish the number of distinct rows
  if (n_unique_out && blockIdx.x == 0 && threadIdx.x == 0) *n_unique_out = (int64_t)*a.n_unique;
}

template <int LPR>
static int launch_bwd(const BwdArgs& a, int64_t* n_unique_out, cudaStream_t st) {
  const int64_t nchunks = (a.n + kChunk - 1) / kChunk;
  const int64_t vchunks = a.perm_G > 1 ? a.perm_M * a.perm_G : nchunks;   // virtual chunks (>= nchunks)
  const unsigned rgrid = (unsigned)((vchunks + 7) / 8);
  if (a.mode == kModeEmit)
    embed_bwd_reduce_kernel<LPR, kModeEmit><<<rgrid, 256, 0, st>>>(a);
  else if (a.mode == kModeBag)
    embed_bwd_reduce_kernel<LPR, kModeBag><<<rgrid, 256, 0, st>>>(a);
  else if (a.mode == kModeBagEmit)
    embed_bwd_reduce_kernel<LPR, kModeBagEmit><<<rgrid, 256, 0, st>>>(a);
  else
    embed_bwd_reduce_kernel<LPR, kModeLocal><<<rgrid, 256, 0, st>>>(a);
  constexpr int NG = 256 / LPR;
  embed_bwd_finish_kernel<LPR><<<(unsigned)((nchunks + NG - 1) / NG), 256, 0, st>>>(a, n_unique_out);
  return launched("embed_bwd_reduce_update", 2);
}

// ------------------------------------------------------------------------------------------
// One-row fields.  A numeric ("dense") feature is a field whose table has a single row scaled by
// feature_value (weighted-column semantics, dataset/SequenceTensorFlowDataset/test4.py:50-55), so
// every sample looks up the same row: no sort is needed, the row's gradient is a column sum over
// the batch.  Warps stride over samples and keep one accumulator per field (LPR lanes per field);
// warps, then CTAs, are combined in a fixed order and the finish kernel applies the update.
// Each term is formed in fp32 in the oracle's evaluation order; the B-term column sum is carried in
// fp64 (thread -> warp -> CTA -> grid, fixed order) and rounded to fp32 once: a 65 536-term fp32 sum
// whose result lands near zero otherwise leaves ~3e-5 absolute on G, which Adagrad's lr/sqrt(0.1)
// slope turns into > 5e-6 on the row (round-1 full-size parity failure).
constexpr int kOneRowPasses = 4;   // fields per launch = kOneRowPasses * 32 / LPR
constexpr int kOneRowCtas = kOneRowCtasMax;
constexpr int kOneRowMax = 64;     // one-row fields per call

struct OneRowArgs {
  float* table = nullptr;
  float* accum = nullptr;
  int64_t row_stride = 0;
  float* lin = nullptr;
  float* lin_accum = nullptr;
  int64_t lin_stride = 0;
  const int64_t* idx = nullptr;
  const float* val = nullptr;
  const int64_t* field_offset = nullptr;
  const float* g_first = nullptr;
  const float* g_fm = nullptr;
  const float* S = nullptr;
  const float* u = nullptr;
  const int32_t* fields = nullptr;
  int64_t B = 0;
  int F = 0;
  int opt = DIR_OPT_SGD;
  float lr = 0.f;
  double* part = nullptr;  // [kOneRowCtas][kOneRowMax][K + 4]
  int* flags = nullptr;    // [kOneRowMax] some sample had a surviving lookup
  unsigned long long* n_unique = nullptr;
  LinOpt lo{};
  float clip = 0.f;        // > 0: tf.clip_by_norm of the field's gradient (its variable has this one row) before the update
  float l1 = 0.f, l2 = 0.f;  // ProximalAdagrad strengths of the table rows
};

template <int LPR, int P>
__global__ void __launch_bounds__(256, P <= 2 ? 3 : 1)
embed_bwd_onerow_kernel(const OneRowArgs a, int f0, int nf) {
  constexpr int K = LPR * 4;
  constexpr int SLOTS = 32 / LPR;
  // samples whose loads are in flight together: with the fp64 accumulators four of them cost 134 registers at
  // P = 2 (one CTA per SM, 12 % of the warp slots: profiles/r02_sharded_1gpu_ncu.txt); two fit three CTAs per SM
  constexpr int UN = P <= 2 ? 2 : 4;
  __shared__ double sm4[8][P][32][4];
  __shared__ double sm1[8][P][32];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int sub = lane % LPR, slot = lane / LPR;
  float4 T[P];
  double acc[P][4], acc1[P];
  int fld[P];
  bool any[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int j = p * SLOTS + slot;
    fld[p] = j < nf ? __ldg(a.fields + f0 + j) : -1;
    T[p] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc[p][0] = acc[p][1] = acc[p][2] = acc[p][3] = 0.0;
    acc1[p] = 0.0;
    any[p] = false;
    if (fld[p] >= 0)
      T[p] = *(reinterpret_cast<const float4*>(a.table + __ldg(a.field_offset + fld[p]) * a.row_stride) + sub);
  }
  const int64_t W = (int64_t)gridDim.x * 8;
  for (int64_t b0 = (int64_t)blockIdx.x * 8 + wib; b0 < a.B; b0 += W * UN) {
    float4 Sb[UN], ub[UN][P];
    float g1[UN], g2[UN], v[UN][P];
    bool ok[UN][P];
#pragma unroll
    for (int s = 0; s < UN; ++s) {
      const int64_t b = b0 + s * W < a.B ? b0 + s * W : a.B - 1;  // clamped; masked by `ok` below
      Sb[s] = __ldg(reinterpret_cast<const float4*>(a.S + b * K) + sub);
      g1[s] = __ldg((a.g_first ? a.g_first : a.g_fm) + b);
      g2[s] = __ldg(a.g_fm + b);
    }
    // Loads only, no branches on the nullable pointers and no consumer in between (a NULL array is
    // replaced by a harmless valid address): every load of the UN samples is in flight before the
    // first value is looked at.
    int64_t id[UN][P];
#pragma unroll
    for (int s = 0; s < UN; ++s) {
      const int64_t b = b0 + s * W < a.B ? b0 + s * W : a.B - 1;
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const int64_t pos = b * a.F + (fld[p] >= 0 ? fld[p] : 0);
        v[s][p] = __ldg(a.val ? a.val + pos : a.S);
        id[s][p] = __ldg(a.idx ? a.idx + pos : a.field_offset);
        ub[s][p] = ldg_stream(a.u ? a.u + pos * K + sub * 4 : a.S);
      }
    }
#pragma unroll
    for (int s = 0; s < UN; ++s) {
      const bool live = b0 + s * W < a.B;
      if (!a.g_first) g1[s] = 0.f;
#pragma unroll
      for (int p = 0; p < P; ++p) {
        if (!a.val) v[s][p] = 1.f;
        if (!a.u) ub[s][p] = make_float4(0.f, 0.f, 0.f, 0.f);
        // pruned: id < 0, value <= 0, or id beyond the field's single row
        ok[s][p] = live && fld[p] >= 0 && (!a.idx || id[s][p] == 0) && v[s][p] > 0.f;
      }
    }
#pragma unroll
    for (int s = 0; s < UN; ++s) {  // samples in ascending order
#pragma unroll
      for (int p = 0; p < P; ++p) {
        if (!ok[s][p]) continue;
        const float x = v[s][p], gg = g2[s];
        acc[p][0] += (double)__fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[s].x, __fmul_rn(x, T[p].x))), ub[s][p].x));
        acc[p][1] += (double)__fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[s].y, __fmul_rn(x, T[p].y))), ub[s][p].y));
        acc[p][2] += (double)__fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[s].z, __fmul_rn(x, T[p].z))), ub[s][p].z));
        acc[p][3] += (double)__fmul_rn(x, __fadd_rn(__fmul_rn(gg, __fsub_rn(Sb[s].w, __fmul_rn(x, T[p].w))), ub[s][p].w));
        acc1[p] += (double)__fmul_rn(g1[s], x);
        any[p] = true;
      }
    }
  }
#pragma unroll
  for (int p = 0; p < P; ++p) {
#pragma unroll
    for (int c = 0; c < 4; ++c) sm4[wib][p][lane][c] = acc[p][c];
    sm1[wib][p][lane] = acc1[p];
    if (any[p] && sub == 0) a.flags[f0 + p * SLOTS + slot] = 1;  // benign race: everyone writes 1
  }
  __syncthreads();
  if (wib < P) {  // warp p adds the 8 warps' sums of pass p in warp order
    const int p = wib;
    const int j = p * SLOTS + slot;
    if (j < nf) {
      double t[4] = {sm4[0][p][lane][0], sm4[0][p][lane][1], sm4[0][p][lane][2], sm4[0][p][lane][3]};
      double t1 = sm1[0][p][lane];
#pragma unroll
      for (int w = 1; w < 8; ++w) {
#pragma unroll
        for (int c = 0; c < 4; ++c) t[c] += sm4[w][p][lane][c];
        t1 += sm1[w][p][lane];
      }
      double* dst = a.part + ((int64_t)blockIdx.x * kOneRowMax + f0 + j) * (K + 4);
#pragma unroll
      for (int c = 0; c < 4; ++c) dst[sub * 4 + c] = t[c];
      if (sub == 0) dst[K] = t1;
    }
  }
}

// One-row field j: 32 component lanes x 8 "g-lanes" of the CTA sum the `ctas` CTA partials in a fixed order;
// tot[c] (c <= K) receives the column sum, rounded to fp32 once.  Every thread of the CTA calls it.
template <int K>
__device__ __forceinline__ void onerow_sum(const double* part, int j, int ctas, float* tot) {
  __shared__ double red[8][33];
  const int cx = threadIdx.x & 31, gy = threadIdx.x >> 5;
  for (int c0 = 0; c0 <= K; c0 += 32) {
    const int c = c0 + cx;
    double t = 0.0;
    if (c <= K)
#pragma unroll 8
      for (int g = gy; g < ctas; g += 8) t += __ldg(part + ((int64_t)g * kOneRowMax + j) * (K + 4) + c);
    red[gy][cx] = t;
    __syncthreads();
    if (gy == 0 && c <= K) {
      double v = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) v += red[k][cx];
      tot[c] = (float)v;  // the one rounding of the column sum
    }
    __syncthreads();
  }
}

// one CTA per one-row field: the column sum, then the row update
template <int LPR>
__global__ void __launch_bounds__(256) embed_bwd_onerow_finish_kernel(const OneRowArgs a, int G) {
  constexpr int K = LPR * 4;
  __shared__ float tot[K + 1];
  const int j = blockIdx.x;
  if (a.flags[j] == 0) return;  // no surviving lookup: the row is not touched
  onerow_sum<K>(a.part, j, G, tot);
  if (a.clip > 0.f) {  // values * clip / max(||values||, clip), the row and the linear weight each a variable
    if (threadIdx.x == 0) {
      double sq = 0.0;
      for (int c = 0; c < K; ++c) sq += (double)tot[c] * tot[c];
      const float den = fmaxf((float)sqrt(sq), a.clip), den1 = fmaxf(fabsf(tot[K]), a.clip);
      for (int c = 0; c < K; ++c) tot[c] = __fdiv_rn(__fmul_rn(tot[c], a.clip), den);
      tot[K] = __fdiv_rn(__fmul_rn(tot[K], a.clip), den1);
    }
    __syncthreads();
  }
  const bool adagrad = a.opt != DIR_OPT_SGD;
  const RowRule rr{a.opt, a.lr, a.l1, a.l2};
  const int64_t row = a.field_offset[a.fields[j]];
  if (threadIdx.x < K) {
    float* tp = a.table + row * a.row_stride + threadIdx.x;
    float acc = 0.f;
    float* ap = nullptr;
    if (adagrad) {
      ap = a.accum + row * a.row_stride + threadIdx.x;
      acc = *ap;
    }
    *tp = upd_rule(*tp, tot[threadIdx.x], acc, rr);
    if (adagrad) *ap = acc;
  } else if (threadIdx.x == K) {
    if (a.lin != nullptr) {
      const int64_t off = row * a.lin_stride;
      float n1, z1;
      lin_load(a.lo, a.lin_accum, off, n1, z1);
      lin_apply(a.lo, a.lin + off, a.lin_accum + off, a.lo.z + off, a.lin[off], n1, z1, tot[K]);
    }
    if (a.n_unique) atomicAdd(a.n_unique, 1ull);
  }
}

template <int LPR>
static int launch_onerow_partials(const OneRowArgs& a, int n_fields, cudaStream_t st, int* ctas) {
  constexpr int PER = kOneRowPasses * (32 / LPR);
  constexpr int SLOTS = 32 / LPR;
  const int64_t want = (a.B + 7) / 8;
  const int G = (int)(want < kOneRowCtas ? want : kOneRowCtas);
  int n = 0;
  *ctas = G;
  if (G == 0) return 0;  // an empty batch on this rank: the emit kernel ships zeros, `touched` = 0
  for (int f0 = 0; f0 < n_fields; f0 += PER, ++n) {
    const int nf = n_fields - f0 < PER ? n_fields - f0 : PER;
    switch ((nf + SLOTS - 1) / SLOTS) {
      case 1: embed_bwd_onerow_kernel<LPR, 1><<<G, 256, 0, st>>>(a, f0, nf); break;
      case 2: embed_bwd_onerow_kernel<LPR, 2><<<G, 256, 0, st>>>(a, f0, nf); break;
      case 3: embed_bwd_onerow_kernel<LPR, 3><<<G, 256, 0, st>>>(a, f0, nf); break;
      default: embed_bwd_onerow_kernel<LPR, 4><<<G, 256, 0, st>>>(a, f0, nf); break;
    }
  }
  return launched("embed_bwd_onerow_partials", n);
}

template <int LPR>
static int launch_onerow(const OneRowArgs& a, int n_fields, cudaStream_t st) {
  int ctas = 0;
  if (int rc = launch_onerow_partials<LPR>(a, n_fields, st, &ctas)) return rc;
  embed_bwd_onerow_finish_kernel<LPR><<<n_fields, 256, 0, st>>>(a, ctas);
  return launched("embed_bwd_onerow");
}

__global__ void publish_count_kernel(const unsigned long long* src, int64_t* dst) { *dst = (int64_t)*src; }

// position / F == (position * magic) >> shift, exact for positions < 2^31:
// shift = 31 + ceil(log2 F), magic = ceil(2^shift / F) <= 2^32 - 1
static void set_div(BwdArgs& a, int F) {
  int lg = 0;
  while ((1 << lg) < F) ++lg;
  a.div_shift = 31 + lg;
  a.div_magic = (uint32_t)((((uint64_t)1 << a.div_shift) + (uint64_t)F - 1) / (uint64_t)F);
}

// The sorted list of n entries that the sort step left in w; an entry's sample is its position / per_sample.
static void set_sorted(BwdArgs& a, const BwdWorkspace& w, int64_t n, int F, int per_sample) {
  a.keys = w.keys;
  a.pos = w.pos;
  a.part = w.part;
  a.part1 = w.part1;
  a.long_list = w.long_list;
  a.long_count = w.long_count;
  a.n_unique = w.n_unique;
  a.n = n;
  a.F = F;
  set_div(a, per_sample);
}

// The emit modes' sums go straight into the owners' buffers of a peer layout (after set_sorted: perm_M needs n).
static void set_peer_emit(BwdArgs& a, const dir_peer_layout& L, const int64_t* owner_off, float* g1_local) {
  a.emit_seg = owner_off;
  a.emit_peers = L.peer_base;
  a.emit_byte_off = L.off_g;
  a.emit_dst_row = (int64_t)L.rank * L.seg_cap;
  a.emit_seg_cap = L.seg_cap;
  a.emit_g1 = g1_local;
  a.emit_G = L.G;
  a.perm_G = L.G;
  a.perm_rank = L.rank;
  a.perm_M = ((a.n + kChunk - 1) / kChunk + L.G - 1) / L.G;
}

// f(std::integral_constant<int, LPR>()) with LPR = K / 4 lanes per K-vector; every caller has checked that K is one
// of 4, 8, 16, 32, 64.
template <class Fn>
static int with_lpr(int K, Fn&& f) {
  switch (K) {
    case 4: return f(std::integral_constant<int, 1>());
    case 8: return f(std::integral_constant<int, 2>());
    case 16: return f(std::integral_constant<int, 4>());
    case 32: return f(std::integral_constant<int, 8>());
    default: return f(std::integral_constant<int, 16>());
  }
}

static int dispatch_bwd(const BwdArgs& a, int K, int64_t* n_unique_out, cudaStream_t st) {
  return with_lpr(K, [&](auto lpr) { return launch_bwd<lpr>(a, n_unique_out, st); });
}

}  // namespace dir

extern "C" size_t dir_embed_bwd_workspace_bytes(int64_t n_lookups, int K) {
  if (n_lookups <= 0 || K <= 0) return 0;
  return dir::carve(nullptr, n_lookups, K).total;
}

extern "C" int dir_embed_bwd_sorted(const void* workspace, int64_t n_lookups,
                                    const uint32_t** sorted_keys, const uint32_t** sorted_pos) {
  using namespace dir;
  if (!workspace || n_lookups <= 0 || !sorted_keys || !sorted_pos)
    return fail(DIR_EINVAL, "embed_bwd_sorted: workspace, n_lookups > 0 and both outputs are required");
  BwdWorkspace w = carve(const_cast<void*>(workspace), n_lookups, 4);
  *sorted_keys = w.keys;
  *sorted_pos = w.pos;
  return 0;
}

extern "C" int dir_embed_bwd_sort(const uint32_t* sort_keys, int64_t n_lookups, int64_t n_rows,
                                  void* workspace, size_t workspace_bytes, dir_stream_t stream) {
  using namespace dir;
  if (n_lookups < 0 || n_lookups >= 0x7fffffffLL)
    return fail(DIR_EINVAL, "embed_bwd_sort: 0 <= n_lookups < 2^31 required");
  if (n_rows <= 0 || n_rows >= 0xffffffffLL)
    return fail(DIR_EINVAL, "embed_bwd_sort: 0 < n_rows < 2^32-1 required");
  if (n_lookups == 0) return 0;
  if (!sort_keys || !workspace) return fail(DIR_EINVAL, "embed_bwd_sort: null pointer");
  // K only sizes the tail of the workspace; the sort part does not depend on it
  BwdWorkspace w = carve(workspace, n_lookups, 4);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "embed_bwd_sort: workspace too small");
  int end_bit = 1;
  while (end_bit < 32 && (((uint64_t)n_rows) >> end_bit) != 0) ++end_bit;  // n_rows itself is a key
  // the hand-written sort (radix.cuh): three small kernels per 8-bit pass, positions implied by the input order
  const int launches = radix_sort_pairs(sort_keys, n_lookups, end_bit, w.keys, w.pos, w.alt_keys, w.pos_in,
                                        w.radix_hist, w.long_count, w.n_unique, static_cast<cudaStream_t>(stream));
  return launched("embed_bwd_sort", launches);
}

namespace dir {
// dir_shard_keys and the sort's first counting pass in one kernel: a CTA forms the keys of one radix tile (2 048
// consecutive entries, coalesced rounds of 256) and counts their low digit while they are in registers.
__global__ void __launch_bounds__(256)
keys_count_kernel(const KeyArgs a, uint32_t* __restrict__ keys, int64_t tiles, uint32_t* __restrict__ hist,
                  uint32_t* zero_a, unsigned long long* zero_b) {
  __shared__ uint32_t sh[256];
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // counters of the consumer of the sorted list start at zero
    *zero_a = 0u;
    *zero_b = 0ull;
  }
  sh[threadIdx.x] = 0u;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kRadixTile;
  // (sample, selected field) of this thread's first entry; a round later the entry is 256 further on: one division
  // per thread instead of two per key
  const uint32_t ns = (uint32_t)a.n_sel;
  uint32_t b = (uint32_t)(base + threadIdx.x) / ns;
  uint32_t j = (uint32_t)(base + threadIdx.x) - b * ns;
  const uint32_t db = 256u / ns, dj = 256u - db * ns;
#pragma unroll
  for (int r = 0; r < kRadixRounds; ++r) {
    const int64_t o = base + r * 256 + threadIdx.x;
    if (o < a.n) {
      const uint32_t key = make_key_bj(a, o, b, (int)j);
      keys[o] = key;
      // plain shared-memory atomics: the input order mixes fields and samples, so lanes rarely meet on a digit
      atomicAdd(&sh[key & 255u], 1u);
    }
    b += db;
    j += dj;
    if (j >= ns) {
      j -= ns;
      ++b;
    }
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * tiles + blockIdx.x] = sh[threadIdx.x];
}
}  // namespace dir

/* dir_shard_keys + dir_embed_bwd_sort in one call: the key kernel counts the first radix digit while the keys
 * are in registers, so the sort starts without a pass of its own over them. */
extern "C" int dir_shard_keys_sort(const int64_t* feature_index, const float* feature_value,
                                   const int64_t* field_offset, const int64_t* field_rows, int64_t n_rows,
                                   int64_t B, int F, int G, const int32_t* field_sel, int n_sel, uint32_t* keys,
                                   int* oob_flag, void* workspace, size_t workspace_bytes, dir_stream_t stream) {
  using namespace dir;
  KeyArgs a;
  if (int rc = key_args("shard_keys_sort", feature_index, feature_value, field_offset, field_rows, n_rows, B, F, G,
                        field_sel, n_sel, oob_flag, a))
    return rc;
  const int64_t n = a.n;
  const int64_t n_keys = G > 1 ? a.cap * G : n_rows;  // the pruned key; every other key is below it
  if (n == 0) {  // nothing to fuse: the two calls
    if (int rc = dir_shard_keys(feature_index, feature_value, field_offset, field_rows, n_rows, B, F, G, field_sel,
                                n_sel, keys, oob_flag, stream))
      return rc;
    return dir_embed_bwd_sort(keys, n, n_keys, workspace, workspace_bytes, stream);
  }
  if (!keys || !workspace) return fail(DIR_EINVAL, "shard_keys_sort: null pointer");
  BwdWorkspace w = carve(workspace, n, 4);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "shard_keys_sort: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int end_bit = 1;
  while (end_bit < 32 && (((uint64_t)n_keys) >> end_bit) != 0) ++end_bit;  // n_keys itself is a key
  const int64_t tiles = radix_tiles(n);
  keys_count_kernel<<<(unsigned)tiles, 256, 0, st>>>(a, keys, tiles, w.radix_hist, w.long_count, w.n_unique);
  const int launches = radix_sort_pairs(keys, n, end_bit, w.keys, w.pos, w.alt_keys, w.pos_in, w.radix_hist,
                                        w.long_count, w.n_unique, st, /*counted=*/true);
  return launched("shard_keys_sort", launches + 1);
}

extern "C" int dir_embed_bwd_reduce_update(
    float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
    const int64_t* feature_index, const float* feature_value, const int64_t* field_offset,
    const float* g_first, const float* g_fm, const float* S, const float* u, int64_t B, int F, int K,
    int64_t n_rows, const int32_t* field_sel, int n_sel, const int32_t* onerow_fields, int n_onerow,
    int optimizer, float lr, const dir_table_opt* table_opt, const dir_linear_opt* linear_opt, void* workspace,
    size_t workspace_bytes, int64_t* n_unique_out, dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0) return fail(DIR_EINVAL, "embed_bwd_reduce_update: B >= 0, F > 0 required");
  if (B * F >= 0x7fffffffLL) return fail(DIR_EINVAL, "embed_bwd_reduce_update: B*F must be < 2^31");
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD && optimizer != DIR_OPT_PROXIMAL_ADAGRAD)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: unknown optimizer");
  if (!table || !g_fm || !S || !workspace)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: table, g_fm, S, workspace are required");
  if (optimizer != DIR_OPT_SGD && !accum)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: Adagrad needs accum");
  const float tl1 = table_opt ? table_opt->l1 : 0.f, tl2 = table_opt ? table_opt->l2 : 0.f;
  if (tl1 < 0.f || tl2 < 0.f) return fail(DIR_EINVAL, "embed_bwd_reduce_update: l1, l2 must be >= 0");
  LinOpt lo;
  if (int rc = resolve_lin("embed_bwd_reduce_update", linear_opt, optimizer, lr, lin, lin_accum, lo)) return rc;
  if (lin && !g_first) return fail(DIR_EINVAL, "embed_bwd_reduce_update: lin needs g_first");
  if (row_stride < K || (row_stride & 3))
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: row_stride must be >= K, multiple of 4");
  if (!aligned16(table) || !aligned16(accum) || !aligned16(S) || !aligned16(u))
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: table, accum, S, u must be 16-byte aligned");
  if (n_rows <= 0 || n_rows >= 0xffffffffLL)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: 0 < n_rows < 2^32-1 required");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: K must be one of 4, 8, 16, 32, 64");
  if (field_sel == nullptr) n_sel = F;
  if (n_sel < 0 || n_sel > F || n_onerow < 0 || n_onerow > kOneRowMax || (n_onerow > 0 && !onerow_fields))
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: need 0 <= n_sel <= F and 0 <= n_onerow <= 64");
  if (n_onerow > 0 && !field_offset)
    return fail(DIR_EINVAL, "embed_bwd_reduce_update: one-row fields need field_offset");
  if (B == 0) return 0;
  const int64_t n = B * n_sel;  // entries the sort step left in the workspace
  BwdWorkspace w = carve(workspace, n > 0 ? n : 1, K);
  if (workspace_bytes < w.total)
    return fail(DIR_ENOMEM, "embed_bwd_reduce_update: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n == 0) cudaMemsetAsync(w.n_unique, 0, 8, st);  // no sort ran: nobody zeroed the counter
  if (n_onerow > 0) {
    cudaMemsetAsync(w.onerow_flags, 0, kOneRowMax * 4, st);
    OneRowArgs o;
    o.table = table; o.accum = accum; o.row_stride = row_stride;
    o.lin = lin; o.lin_accum = lin_accum; o.lin_stride = lin_stride; o.lo = lo;
    o.idx = feature_index; o.val = feature_value; o.field_offset = field_offset; o.fields = onerow_fields;
    o.g_first = g_first; o.g_fm = g_fm; o.S = S; o.u = u; o.B = B; o.F = F;
    o.opt = optimizer; o.lr = lr; o.l1 = tl1; o.l2 = tl2;
    o.part = w.onerow_part; o.flags = w.onerow_flags; o.n_unique = w.n_unique;
    if (int rc = with_lpr(K, [&](auto lpr) { return launch_onerow<lpr>(o, n_onerow, st); })) return rc;
  }
  if (n == 0) {
    if (n_unique_out) {
      publish_count_kernel<<<1, 1, 0, st>>>(w.n_unique, n_unique_out);
      return launched("embed_bwd_reduce_update/count");
    }
    return 0;
  }
  BwdArgs a;
  set_sorted(a, w, n, F, n_sel);
  a.mode = kModeLocal;
  a.table = table; a.accum = accum; a.row_stride = row_stride;
  a.lin = lin; a.lin_accum = lin_accum; a.lin_stride = lin_stride; a.lo = lo;
  a.val = feature_value; a.g_first = g_first; a.g_fm = g_fm; a.S = S; a.u = u;
  a.field_sel = field_sel; a.n_sel = n_sel;
  a.pruned_key = (uint32_t)n_rows; a.opt = optimizer; a.lr = lr; a.l1 = tl1; a.l2 = tl2;
  return dispatch_bwd(a, K, n_unique_out, st);
}

/* requester side of a row-sharded table: per-unique-row gradient sums -> gu, or (layout != NULL) straight
 * into the owners' buffers over NVLink (include/dir_b200.h) */
static int reduce_emit(const char* what, const float* ubuf, int64_t ubuf_stride, const float* feature_value,
                       const float* g_first, const float* g_fm, const float* S, const float* u,
                       const uint32_t* uidx, int64_t B, int F, int K, int64_t n_keys, float* gu,
                       int64_t gu_stride, const dir_peer_layout* layout, const int64_t* owner_off, float* g1_local,
                       void* workspace, size_t workspace_bytes, dir_stream_t stream, const int32_t* field_sel,
                       int n_sel, int read_key = 0) {
  using namespace dir;
  if (B < 0 || F <= 0) return fail(DIR_EINVAL, "%s: B >= 0, F > 0 required", what);
  if (field_sel == nullptr) n_sel = F;      // the sorted list covers every field
  if (n_sel < 0 || n_sel > F) return fail(DIR_EINVAL, "%s: 0 <= n_sel <= F required", what);
  const int64_t n = B * n_sel;
  if (n >= 0x7fffffffLL) return fail(DIR_EINVAL, "%s: B*F must be < 2^31", what);
  if (n == 0) return 0;
  if (!ubuf || !g_fm || !S || !uidx || !workspace || (!gu && !layout))
    return fail(DIR_EINVAL, "%s: ubuf, g_fm, S, uidx, workspace and a destination are required", what);
  if (layout && (!owner_off || !g1_local)) return fail(DIR_EINVAL, "%s: owner_off and g1_local are required", what);
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "%s: K must be one of 4, 8, 16, 32, 64", what);
  if (ubuf_stride < K || (ubuf_stride & 3) || (gu && (gu_stride < K + 1 || (gu_stride & 3))))
    return fail(DIR_EINVAL, "%s: strides must be multiples of 4, >= K (ubuf), >= K+1 (gu)", what);
  if (!aligned16(ubuf) || !aligned16(gu) || !aligned16(S) || !aligned16(u))
    return fail(DIR_EINVAL, "%s: ubuf, gu, S, u must be 16-byte aligned", what);
  if (n_keys <= 0 || n_keys >= 0xffffffffLL) return fail(DIR_EINVAL, "%s: 0 < n_keys < 2^32-1 required", what);
  BwdWorkspace w = carve(workspace, n, K);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "%s: workspace too small", what);
  BwdArgs a;
  set_sorted(a, w, n, F, n_sel);
  a.mode = kModeEmit;
  a.table = const_cast<float*>(ubuf); a.row_stride = ubuf_stride; a.emit_read_key = read_key;
  a.val = feature_value; a.g_first = g_first; a.g_fm = g_fm; a.S = S; a.u = u;
  a.field_sel = field_sel; a.n_sel = n_sel;
  a.pruned_key = (uint32_t)n_keys; a.rowidx = uidx;
  a.emit = gu; a.emit_stride = gu_stride;
  if (layout) set_peer_emit(a, *layout, owner_off, g1_local);
  return dispatch_bwd(a, K, nullptr, static_cast<cudaStream_t>(stream));
}

/* the same per-distinct-row sums for a table that lives HERE (rows read at their global row, sums written to
 * gu[uidx]): the first pass of the clipped backward (csrc/clip.cu) */
extern "C" int dir_embed_bwd_reduce_emit_local(const float* table, int64_t row_stride, const float* feature_value,
                                               const float* g_first, const float* g_fm, const float* S,
                                               const float* u, const uint32_t* uidx, int64_t B, int F, int K,
                                               int64_t n_rows, const int32_t* field_sel, int n_sel, float* gu,
                                               int64_t gu_stride, void* workspace, size_t workspace_bytes,
                                               dir_stream_t stream) {
  if (!gu) return dir::fail(DIR_EINVAL, "embed_bwd_reduce_emit_local: gu is required");
  return reduce_emit("embed_bwd_reduce_emit_local", table, row_stride, feature_value, g_first, g_fm, S, u, uidx, B, F,
                     K, n_rows, gu, gu_stride, nullptr, nullptr, nullptr, workspace, workspace_bytes, stream,
                     field_sel, n_sel, 1);
}

extern "C" int dir_embed_bwd_reduce_emit_to(const dir_peer_layout* layout, const float* feature_value,
                                            const float* g_first, const float* g_fm, const float* S,
                                            const float* u, const uint32_t* uidx, const int64_t* owner_off,
                                            int64_t B, int F, int64_t n_keys, const int32_t* field_sel,
                                            int n_sel, float* g1_local, void* workspace,
                                            size_t workspace_bytes, dir_stream_t stream) {
  using namespace dir;
  if (!layout || !layout->peer_base || !layout->local || layout->G <= 0 || layout->G > 64)
    return fail(DIR_EINVAL, "embed_bwd_reduce_emit_to: a filled dir_peer_layout is required");
  const float* rows = reinterpret_cast<const float*>(layout->local + layout->off_rows);
  return reduce_emit("embed_bwd_reduce_emit_to", rows, layout->K, feature_value, g_first, g_fm, S, u, uidx, B, F,
                     layout->K, n_keys, nullptr, 0, layout, owner_off, g1_local, workspace, workspace_bytes, stream,
                     field_sel, n_sel);
}

/* multi-hot bags: backward + fused update on the sorted (row, entry) list (include/dir_b200.h) */
extern "C" int dir_embed_bag_bwd_reduce_update(
    float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
    const float* bag_weight, const uint32_t* entry_slot, const float* entry_x, int64_t nnz, const float* emb,
    const float* g_first, const float* g_fm, const float* S, const float* u, int64_t B, int F, int K,
    int64_t n_rows, int optimizer, float lr, const dir_linear_opt* linear_opt, void* workspace,
    size_t workspace_bytes, int64_t* n_unique_out, dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0 || nnz < 0 || nnz >= 0x7fffffffLL || B * F >= 0x7fffffffLL)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: B >= 0, F > 0, 0 <= nnz < 2^31, B*F < 2^31 required");
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: unknown optimizer");
  if (optimizer == DIR_OPT_ADAGRAD && !accum)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: Adagrad needs accum");
  LinOpt lo;
  if (int rc = resolve_lin("embed_bag_bwd_reduce_update", linear_opt, optimizer, lr, lin, lin_accum, lo)) return rc;
  if (lin && !g_first) return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: lin needs g_first");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: K must be one of 4, 8, 16, 32, 64");
  if (row_stride < K || (row_stride & 3))
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: row_stride must be >= K, multiple of 4");
  if (n_rows <= 0 || n_rows >= 0xffffffffLL)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: 0 < n_rows < 2^32-1 required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B == 0 || nnz == 0) {
    if (n_unique_out) cudaMemsetAsync(n_unique_out, 0, 8, st);
    return 0;
  }
  if (!table || !entry_slot || !entry_x || !emb || !g_fm || !S || !workspace)
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: table, entry_slot, entry_x, emb, g_fm, S, workspace are required");
  if (!aligned16(table) || !aligned16(accum) || !aligned16(S) || !aligned16(u) || !aligned16(emb))
    return fail(DIR_EINVAL, "embed_bag_bwd_reduce_update: table, accum, S, u, emb must be 16-byte aligned");
  BwdWorkspace w = carve(workspace, nnz, K);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "embed_bag_bwd_reduce_update: workspace too small");
  BwdArgs a;
  set_sorted(a, w, nnz, F, F);
  a.mode = kModeBag;
  a.table = table; a.accum = accum; a.row_stride = row_stride;
  a.lin = lin; a.lin_accum = lin_accum; a.lin_stride = lin_stride; a.lo = lo;
  a.val = bag_weight; a.g_first = g_first; a.g_fm = g_fm; a.S = S; a.u = u;
  a.entry_slot = entry_slot; a.entry_x = entry_x; a.emb = emb;
  a.pruned_key = (uint32_t)n_rows; a.opt = optimizer; a.lr = lr;
  return dispatch_bwd(a, K, n_unique_out, st);
}

/* Bags through a row-sharded table, requester side: the per-entry gradients of dir_embed_bag_bwd_reduce_update,
 * summed per distinct row and stored straight into the owners' buffers like dir_embed_bwd_reduce_emit_to does
 * (the sorted list = the entries' composite keys, dir_shard_bag_keys + dir_embed_bwd_sort; uidx / owner_off from
 * dir_shard_unique).  No row is read: an entry's gradient needs only the bag's combined embedding. */
extern "C" int dir_embed_bag_bwd_reduce_emit_to(const dir_peer_layout* layout, const float* bag_weight,
                                                const uint32_t* entry_slot, const float* entry_x, int64_t nnz,
                                                const float* emb, const float* g_first, const float* g_fm,
                                                const float* S, const float* u, const uint32_t* uidx,
                                                const int64_t* owner_off, int64_t B, int F, int64_t n_keys,
                                                float* g1_local, void* workspace, size_t workspace_bytes,
                                                dir_stream_t stream) {
  using namespace dir;
  const char* what = "embed_bag_bwd_reduce_emit_to";
  if (!layout || !layout->peer_base || !layout->local || layout->G <= 0 || layout->G > 64)
    return fail(DIR_EINVAL, "%s: a filled dir_peer_layout is required", what);
  const int K = layout->K;
  if (B < 0 || F <= 0 || nnz < 0 || nnz >= 0x7fffffffLL || B * F >= 0x7fffffffLL)
    return fail(DIR_EINVAL, "%s: B >= 0, F > 0, 0 <= nnz < 2^31, B*F < 2^31 required", what);
  if (B == 0 || nnz == 0) return 0;
  if (!entry_slot || !entry_x || !emb || !g_fm || !S || !uidx || !owner_off || !g1_local || !workspace)
    return fail(DIR_EINVAL, "%s: entry_slot, entry_x, emb, g_fm, S, uidx, owner_off, g1_local, workspace are required",
                what);
  if (!aligned16(S) || !aligned16(u) || !aligned16(emb))
    return fail(DIR_EINVAL, "%s: S, u, emb must be 16-byte aligned", what);
  if (n_keys <= 0 || n_keys >= 0xffffffffLL) return fail(DIR_EINVAL, "%s: 0 < n_keys < 2^32-1 required", what);
  BwdWorkspace w = carve(workspace, nnz, K);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "%s: workspace too small", what);
  BwdArgs a;
  set_sorted(a, w, nnz, F, F);
  a.mode = kModeBagEmit;
  a.row_stride = K;
  a.val = bag_weight; a.g_first = g_first; a.g_fm = g_fm; a.S = S; a.u = u;
  a.entry_slot = entry_slot; a.entry_x = entry_x; a.emb = emb;
  a.pruned_key = (uint32_t)n_keys; a.rowidx = uidx;
  set_peer_emit(a, *layout, owner_off, g1_local);
  return dispatch_bwd(a, K, nullptr, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------
// Row-sharded tables: one-row (numeric) fields are REPLICATED parameters.  Every sample of every rank
// hits the same row, so sorting / exchanging those lookups (a third of cfg2's) buys nothing: each rank
// forms the field's gradient over its own samples (the column-sum kernel above), the G partial sums meet
// in every rank's exchange buffer, and after the step's barrier every rank adds them in rank order and
// applies the same update to its replica (csrc/shard_peer.cu: dir_shard_dense_apply).
namespace dir {

struct OneRowWs {
  int* flags;    // [kOneRowMax]
  double* part;  // [kOneRowCtas][kOneRowMax][K + 4]
  size_t total;
};
static OneRowWs onerow_carve(void* base, int K) {
  OneRowWs w;
  char* p = static_cast<char*>(base);
  w.flags = reinterpret_cast<int*>(p);
  const size_t off = align_up((size_t)kOneRowMax * 4, 256);
  w.part = reinterpret_cast<double*>(p ? p + off : nullptr);
  w.total = off + align_up((size_t)kOneRowCtas * kOneRowMax * (K + 4) * 8, 256);
  return w;
}

// one CTA per one-row field: the column sum of embed_bwd_onerow_finish_kernel, then the field's
// (G[K], g1, touched, 0, 0) is stored into dense[rank][j] of EVERY rank's exchange buffer
template <int LPR>
__global__ void __launch_bounds__(256)
onerow_emit_to_kernel(const OneRowArgs a, int ctas, const dir_peer_layout L) {
  constexpr int K = LPR * 4;
  __shared__ __align__(16) float tot[K + 4];
  const int j = blockIdx.x;
  onerow_sum<K>(a.part, j, ctas, tot);
  if (threadIdx.x == 0) {
    tot[K + 1] = a.flags[j] != 0 ? 1.f : 0.f;  // some sample of this rank had a surviving lookup
    tot[K + 2] = tot[K + 3] = 0.f;
  }
  __syncthreads();
  constexpr int NV = LPR + 1;  // float4s per row
  const int64_t row = (int64_t)L.rank * L.n_dense + j;
  for (int t = threadIdx.x; t < L.G * NV; t += blockDim.x) {
    const int q = t / NV, v = t % NV;
    float4* dst = reinterpret_cast<float4*>(__ldg(L.peer_base + q) + L.off_dense) + row * NV + v;
    *dst = *reinterpret_cast<const float4*>(tot + 4 * v);
  }
}

}  // namespace dir

extern "C" size_t dir_shard_dense_workspace_bytes(int K) {
  if (K <= 0) return 0;
  return dir::onerow_carve(nullptr, K).total;
}

extern "C" int dir_shard_dense_emit(const dir_peer_layout* layout, const float* dense_table, int64_t row_stride,
                                    const int64_t* feature_index, const float* feature_value,
                                    const int64_t* dense_field_offset, const float* g_first, const float* g_fm,
                                    const float* S, const float* u, const int32_t* onerow_fields, int64_t B, int F,
                                    void* workspace, size_t workspace_bytes, dir_stream_t stream) {
  using namespace dir;
  if (!layout || !layout->peer_base || layout->G <= 0 || layout->G > 64 || layout->rank < 0 || layout->rank >= layout->G)
    return fail(DIR_EINVAL, "shard_dense_emit: a filled dir_peer_layout is required");
  const int K = layout->K, n_onerow = layout->n_dense;
  if (n_onerow == 0) return 0;
  if (B < 0 || F <= 0 || n_onerow < 0 || n_onerow > kOneRowMax)
    return fail(DIR_EINVAL, "shard_dense_emit: B >= 0, F > 0, 0 <= n_dense <= 64 required");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "shard_dense_emit: K must be one of 4, 8, 16, 32, 64");
  if (!dense_table || !dense_field_offset || (B > 0 && (!g_fm || !S)) || !onerow_fields || !workspace)
    return fail(DIR_EINVAL, "shard_dense_emit: null pointer");
  if (row_stride < K || (row_stride & 3)) return fail(DIR_EINVAL, "shard_dense_emit: row_stride must be >= K, multiple of 4");
  if (!aligned16(dense_table) || !aligned16(S) || !aligned16(u))
    return fail(DIR_EINVAL, "shard_dense_emit: dense_table, S, u must be 16-byte aligned");
  OneRowWs w = onerow_carve(workspace, K);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "shard_dense_emit: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaMemsetAsync(w.flags, 0, kOneRowMax * 4, st);
  OneRowArgs o;
  o.table = const_cast<float*>(dense_table); o.row_stride = row_stride;
  o.idx = feature_index; o.val = feature_value; o.field_offset = dense_field_offset; o.fields = onerow_fields;
  o.g_first = g_first; o.g_fm = g_fm; o.S = S; o.u = u; o.B = B; o.F = F;
  o.part = w.part; o.flags = w.flags;
  return with_lpr(K, [&](auto lpr) {
    int ctas = 0;
    if (int rc = launch_onerow_partials<lpr>(o, n_onerow, st, &ctas)) return rc;
    onerow_emit_to_kernel<lpr><<<n_onerow, 256, 0, st>>>(o, ctas, *layout);
    return launched("shard_dense_emit");
  });
}

extern "C" int dir_embed_bwd_onerow_update(float* table, float* accum, int64_t row_stride, float* lin,
                                           float* lin_accum, int64_t lin_stride, const int64_t* feature_index,
                                           const float* feature_value, const int64_t* field_offset,
                                           const float* g_first, const float* g_fm, const float* S, const float* u,
                                           int64_t B, int F, int K, const int32_t* onerow_fields, int n_onerow,
                                           int optimizer, float lr, const dir_table_opt* table_opt,
                                           const dir_linear_opt* linear_opt, float clip_norm, void* workspace,
                                           size_t workspace_bytes, int64_t* n_unique_out, dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0 || n_onerow < 0 || n_onerow > kOneRowMax || clip_norm < 0.f)
    return fail(DIR_EINVAL, "embed_bwd_onerow_update: B >= 0, F > 0, 0 <= n_onerow <= 64, clip_norm >= 0 required");
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD && optimizer != DIR_OPT_PROXIMAL_ADAGRAD)
    return fail(DIR_EINVAL, "embed_bwd_onerow_update: unknown optimizer");
  const float tl1 = table_opt ? table_opt->l1 : 0.f, tl2 = table_opt ? table_opt->l2 : 0.f;
  if (tl1 < 0.f || tl2 < 0.f) return fail(DIR_EINVAL, "embed_bwd_onerow_update: l1, l2 must be >= 0");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "embed_bwd_onerow_update: K must be one of 4, 8, 16, 32, 64");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_unique_out) cudaMemsetAsync(n_unique_out, 0, 8, st);
  if (B == 0 || n_onerow == 0) return 0;
  if (!table || !g_fm || !S || !workspace || !onerow_fields || !field_offset)
    return fail(DIR_EINVAL, "embed_bwd_onerow_update: table, g_fm, S, workspace, onerow_fields, field_offset are required");
  if (optimizer != DIR_OPT_SGD && !accum) return fail(DIR_EINVAL, "embed_bwd_onerow_update: Adagrad needs accum");
  LinOpt lo;
  if (int rc = resolve_lin("embed_bwd_onerow_update", linear_opt, optimizer, lr, lin, lin_accum, lo)) return rc;
  if (lin && !g_first) return fail(DIR_EINVAL, "embed_bwd_onerow_update: lin needs g_first");
  if (row_stride < K || (row_stride & 3)) return fail(DIR_EINVAL, "embed_bwd_onerow_update: row_stride must be >= K, multiple of 4");
  if (!aligned16(table) || !aligned16(accum) || !aligned16(S) || !aligned16(u))
    return fail(DIR_EINVAL, "embed_bwd_onerow_update: table, accum, S, u must be 16-byte aligned");
  OneRowWs w = onerow_carve(workspace, K);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "embed_bwd_onerow_update: workspace too small");
  cudaMemsetAsync(w.flags, 0, kOneRowMax * 4, st);
  OneRowArgs o;
  o.table = table; o.accum = accum; o.row_stride = row_stride;
  o.lin = lin; o.lin_accum = lin_accum; o.lin_stride = lin_stride; o.lo = lo;
  o.idx = feature_index; o.val = feature_value; o.field_offset = field_offset; o.fields = onerow_fields;
  o.g_first = g_first; o.g_fm = g_fm; o.S = S; o.u = u; o.B = B; o.F = F;
  o.opt = optimizer; o.lr = lr; o.l1 = tl1; o.l2 = tl2; o.clip = clip_norm;
  o.part = w.part; o.flags = w.flags; o.n_unique = reinterpret_cast<unsigned long long*>(n_unique_out);
  return with_lpr(K, [&](auto lpr) { return launch_onerow<lpr>(o, n_onerow, st); });
}
