// K1+K2+K3: multi-field embedding gather fused with the first-order term and the FM
// second-order interaction.  One warp per sample; LPR = K/4 lanes hold one row as float4s, so a
// warp-wide load fetches 32/LPR rows (512 B) and UNR such loads are in flight before any math.
// HBM/latency-bound: no tensor cores (the work is a gather and a per-sample reduction).
//
// Reference math: models/DeepFM/deepFM.py:329-334 (FM), :255-263 (first order), :383-393 (lookup).
#include "common.cuh"

namespace dir {

struct FwdArgs {
  const float* table;
  int64_t row_stride;
  const float* lin;
  int64_t lin_stride;
  const float* bias;
  const int64_t* idx;
  const float* val;
  const int64_t* field_offset;
  const int64_t* field_rows;
  int64_t n_rows;
  int64_t B;
  int F;
  float* emb;
  float* S;
  float* first;
  float* fm;
  uint32_t* sort_keys;
  int* oob_flag;
};

// UNR = 8 asks for three CTAs per SM, the 80 registers it has always had (ptxas otherwise takes 99 and leaves
// two); 0 sets no minimum for the others
template <int LPR, int UNR>
__global__ void __launch_bounds__(256, UNR >= 8 ? 3 : 0) embed_fm_fwd_kernel(const FwdArgs a) {
  constexpr int K = LPR * 4;
  constexpr int RPW = 32 / LPR;  // rows fetched by one warp-wide load
  const int lane = threadIdx.x & 31;
  const int slot = lane / LPR;
  const int sub = lane % LPR;
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= a.B) return;  // whole warp leaves together

  const int F = a.F;
  const int64_t base = b * F;
  const uint32_t pruned_key = (uint32_t)a.n_rows;
  float4 Sv = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 Qv = make_float4(0.f, 0.f, 0.f, 0.f);
  float fo = 0.f;
  const uint64_t pol_keep = policy_evict_last();
  const uint64_t pol_once = policy_evict_first();

  for (int f0 = 0; f0 < F; f0 += RPW * UNR) {
    float4 t[UNR];
    float v[UNR], w[UNR];
    int64_t row[UNR];
    bool keep[UNR];
    // ids, values and field bounds first ...
#pragma unroll
    for (int j = 0; j < UNR; ++j) {
      const int f = f0 + j * RPW + slot;
      const bool active = f < F;
      int64_t id = -1, lo = 0, nf = 0;
      float val = 1.f;
      if (active) {
        id = __ldg(a.idx + base + f);
        if (a.val) val = __ldg(a.val + base + f);
        lo = __ldg(a.field_offset + f);
        nf = a.field_rows ? __ldg(a.field_rows + f) : a.n_rows - lo;
      }
      bool k = active && id >= 0 && val > 0.f;
      if (k && id >= nf) {  // TF's CPU Gather raises here; prune and report
        k = false;
        if (a.oob_flag) *a.oob_flag = 1;
      }
      keep[j] = k;
      row[j] = lo + id;
      v[j] = k ? val : 0.f;
    }
    // ... then every row load of this pass is issued before the first use
#pragma unroll
    for (int j = 0; j < UNR; ++j) {
      t[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      w[j] = 0.f;
      if (keep[j]) {
        // a 64-byte L2 fill and evict_last rows were both measured and change nothing (DESIGN.md section 3)
        t[j] = ldg_hint(a.table + row[j] * a.row_stride + sub * 4, pol_once);
        if (a.lin != nullptr && sub == 0) w[j] = ldg_hint1(a.lin + row[j] * a.lin_stride, pol_keep);
      }
    }
#pragma unroll
    for (int j = 0; j < UNR; ++j) {
      const int f = f0 + j * RPW + slot;
      if (f < F) {
        float4 e;
        e.x = v[j] * t[j].x;
        e.y = v[j] * t[j].y;
        e.z = v[j] * t[j].z;
        e.w = v[j] * t[j].w;
        Sv.x += e.x; Sv.y += e.y; Sv.z += e.z; Sv.w += e.w;
        Qv.x = fmaf(e.x, e.x, Qv.x); Qv.y = fmaf(e.y, e.y, Qv.y);
        Qv.z = fmaf(e.z, e.z, Qv.z); Qv.w = fmaf(e.w, e.w, Qv.w);
        fo = fmaf(v[j], w[j], fo);
        if (a.emb) stg_hint(a.emb + (base + f) * K + sub * 4, e, pol_once);
        if (a.sort_keys && sub == 0)
          a.sort_keys[base + f] = keep[j] ? (uint32_t)row[j] : pruned_key;
      }
    }
  }

  // sum the RPW row slots: lanes with equal `sub` hold the same 4 embedding components
#pragma unroll
  for (int o = LPR; o < 32; o <<= 1) {
    Sv.x += __shfl_xor_sync(0xffffffffu, Sv.x, o);
    Sv.y += __shfl_xor_sync(0xffffffffu, Sv.y, o);
    Sv.z += __shfl_xor_sync(0xffffffffu, Sv.z, o);
    Sv.w += __shfl_xor_sync(0xffffffffu, Sv.w, o);
    Qv.x += __shfl_xor_sync(0xffffffffu, Qv.x, o);
    Qv.y += __shfl_xor_sync(0xffffffffu, Qv.y, o);
    Qv.z += __shfl_xor_sync(0xffffffffu, Qv.z, o);
    Qv.w += __shfl_xor_sync(0xffffffffu, Qv.w, o);
  }
  // 0.5 * sum_k ((sum_f e)^2 - sum_f e^2), deepFM.py:331-333
  float fmv = (Sv.x * Sv.x - Qv.x) + (Sv.y * Sv.y - Qv.y) + (Sv.z * Sv.z - Qv.z) +
              (Sv.w * Sv.w - Qv.w);
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) fmv += __shfl_xor_sync(0xffffffffu, fmv, o);
  fo = warp_sum(fo);

  if (a.S && slot == 0) *reinterpret_cast<float4*>(a.S + b * K + sub * 4) = Sv;
  if (lane == 0) {
    a.fm[b] = 0.5f * fmv;
    if (a.first) a.first[b] = fo + (a.bias ? __ldg(a.bias) : 0.f);
  }
}

template <int LPR>
static int launch_fwd(const FwdArgs& a, cudaStream_t st) {
  constexpr int RPW = 32 / LPR;
  const int iters = (a.F + RPW - 1) / RPW;
  const dim3 block(256);
  const dim3 grid((unsigned)((a.B + 7) / 8));
#define DIR_FWD_CASE(U)                                      \
  embed_fm_fwd_kernel<LPR, U><<<grid, block, 0, st>>>(a); \
  break;
  switch (iters) {
    case 1: DIR_FWD_CASE(1)
    case 2: DIR_FWD_CASE(2)
    case 3: DIR_FWD_CASE(3)
    case 4: DIR_FWD_CASE(4)
    case 5: DIR_FWD_CASE(5)
    case 6: DIR_FWD_CASE(6)
    default: DIR_FWD_CASE(8)
  }
#undef DIR_FWD_CASE
  return launched("embed_fm_fwd");
}

}  // namespace dir

extern "C" int dir_embed_fm_fwd(const float* table, int64_t row_stride, const float* lin,
                                int64_t lin_stride, const float* bias,
                                const int64_t* feature_index, const float* feature_value,
                                const int64_t* field_offset, const int64_t* field_rows,
                                int64_t n_rows, int64_t B, int F, int K, float* emb, float* S,
                                float* first, float* fm, uint32_t* sort_keys, int* oob_flag,
                                dir_stream_t stream) {
  using namespace dir;
  if (B < 0 || F <= 0) return fail(DIR_EINVAL, "embed_fm_fwd: B >= 0 and F > 0 required");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "embed_fm_fwd: K must be one of 4, 8, 16, 32, 64");
  if (B == 0) return 0;  // empty batch: nothing to read or write (pointers may be NULL)
  if (!table || !feature_index || !field_offset || !fm)
    return fail(DIR_EINVAL, "embed_fm_fwd: table, feature_index, field_offset, fm are required");
  if (lin && !first) return fail(DIR_EINVAL, "embed_fm_fwd: `first` is required when `lin` is given");
  if (row_stride < K || (row_stride & 3))
    return fail(DIR_EINVAL, "embed_fm_fwd: row_stride must be >= K and a multiple of 4");
  if (!aligned16(table) || !aligned16(emb) || !aligned16(S))
    return fail(DIR_EINVAL, "embed_fm_fwd: table, emb and S must be 16-byte aligned");
  if (n_rows <= 0 || (sort_keys && n_rows >= 0xffffffffLL))
    return fail(DIR_EINVAL, "embed_fm_fwd: 0 < n_rows (< 2^32-1 when sort_keys is given) required");
  if ((B + 7) / 8 > 0x7fffffffLL) return fail(DIR_EINVAL, "embed_fm_fwd: B too large");
  FwdArgs a{table, row_stride, lin,        lin_stride, bias, feature_index, feature_value,
            field_offset, field_rows, n_rows, B, F, emb, S, first, fm, sort_keys, oob_flag};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (K) {
    case 4: return launch_fwd<1>(a, st);
    case 8: return launch_fwd<2>(a, st);
    case 16: return launch_fwd<4>(a, st);
    case 32: return launch_fwd<8>(a, st);
    case 64: return launch_fwd<16>(a, st);
    default: return fail(DIR_EINVAL, "embed_fm_fwd: K must be one of 4, 8, 16, 32, 64");
  }
}
