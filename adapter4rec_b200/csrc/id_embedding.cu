// ID-embedding item tower (--item_tower id): nn.Embedding(item_num + 1, D, padding_idx=0) as reached from Model.forward
// (`input_embs_all = self.id_embedding(sample_items)`, the IDvs.MoRec branch of Downstream/Text/model/model.py).
//
// Forward: one warp per occurrence row r of ids [B, S1, 2] (flat index r = (b*S1 + j)*2 + t).  The lanes read the fp32
// master row with 128-bit loads, round to bf16 (RNE, as a4r_cast_transpose_f32_bf16) and write emb[r]; when t == 0 and
// j < S1 - 1 the same registers are also written to hist[b, j] (the user-encoder input, which the modal path builds with a
// separate `.contiguous()` copy).  No bf16 copy of the table exists: the bytes moved are R*D*(4 + 2) + B*(S1-1)*D*2.
//
// Backward: the occurrences arrive grouped by id (a stable sort of the ids: `sorted` ascending, `order` the flat
// occurrence indices, ascending inside one id).  One warp per id segment — the warp whose sorted position starts the
// segment — sums the gradient rows of the segment in fp32, in ascending occurrence order, with the d_hist[b, j] term right
// after the d_emb term of an occurrence (b, j, 0), and writes the row once (grad = sum, or grad + sum when accumulating).
// No atomics: the bits depend on the ids only, never on scheduling.  Each lane owns two columns of a 64-column chunk; the
// segment is walked 32 occurrences at a time (one coalesced load of `sorted` / `order`, broadcast by shuffles), so the
// row loads of consecutive occurrences are independent and overlap.
#include "a4r_common.cuh"

namespace {

struct IdFwdParams {
  const float* table;     // [V, D]
  const int64_t* ids;     // [R] = [B, S1, 2]
  __nv_bfloat16* emb;     // [R, D]
  __nv_bfloat16* hist;    // [B, S1 - 1, D] or nullptr
  int64_t R, S1, D, V;
};

__global__ void __launch_bounds__(256) id_embed_gather_kernel(IdFwdParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t nvec = p.D >> 2;
  for (int64_t r = warp; r < p.R; r += nwarps) {
    const int64_t id = p.ids[r];
    const bool valid = id >= 0 && id < p.V;      // an id outside the table reads as a zero row
    const int64_t slot = r >> 1, b = slot / p.S1, j = slot - b * p.S1;
    const bool to_hist = p.hist != nullptr && (r & 1) == 0 && j < p.S1 - 1;
    const float4* src = reinterpret_cast<const float4*>(p.table + (valid ? id : 0) * p.D);
    uint2* dst = reinterpret_cast<uint2*>(p.emb + r * p.D);
    uint2* dst_h = to_hist ? reinterpret_cast<uint2*>(p.hist + (b * (p.S1 - 1) + j) * p.D) : nullptr;
    for (int64_t i = lane; i < nvec; i += 32) {
      const float4 v = valid ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      const uint2 o = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
      dst[i] = o;
      if (to_hist) dst_h[i] = o;
    }
  }
}

struct IdBwdParams {
  const int64_t* sorted;         // [R] ids, ascending
  const int64_t* order;          // [R] flat occurrence index of sorted[k], ascending inside equal ids
  const __nv_bfloat16* d_emb;    // [R, D]
  const __nv_bfloat16* d_hist;   // [B, S1 - 1, D] or nullptr
  float* grad;                   // [V, D]
  int64_t R, S1, D, V, skip_idx;
  int accumulate;
};

__global__ void __launch_bounds__(256) id_embed_bwd_kernel(IdBwdParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t k = warp; k < p.R; k += nwarps) {
    const int64_t id = p.sorted[k];
    if (k > 0 && p.sorted[k - 1] == id) continue;                  // not the start of a segment
    if (id < 0 || id >= p.V || id == p.skip_idx) continue;         // padding row / outside the table: never written
    float* out = p.grad + id * p.D;
    for (int64_t c0 = 0; c0 < p.D; c0 += 64) {
      const int64_t c = c0 + 2 * lane;
      const bool active = c < p.D;
      float2 acc = make_float2(0.f, 0.f);
      for (int64_t k0 = k; k0 < p.R; k0 += 32) {
        const int64_t kk = k0 + lane;
        const bool same = kk < p.R && p.sorted[kk] == id;
        const int64_t rr = same ? p.order[kk] : 0;
        const int n = __popc(__ballot_sync(0xffffffffu, same));   // sorted: the matching lanes are a prefix
#pragma unroll 4
        for (int q = 0; q < n; ++q) {
          const int64_t r = __shfl_sync(0xffffffffu, rr, q);
          if (active) {
            const float2 g = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(p.d_emb + r * p.D + c));
            acc.x += g.x;
            acc.y += g.y;
            const int64_t slot = r >> 1, b = slot / p.S1, j = slot - b * p.S1;
            if (p.d_hist != nullptr && (r & 1) == 0 && j < p.S1 - 1) {
              const float2 h = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(p.d_hist + (b * (p.S1 - 1) + j) * p.D + c));
              acc.x += h.x;
              acc.y += h.y;
            }
          }
        }
        if (n < 32) break;
      }
      if (active) {
        float2* o = reinterpret_cast<float2*>(out + c);
        if (p.accumulate) {
          const float2 prev = *o;
          acc.x = prev.x + acc.x;
          acc.y = prev.y + acc.y;
        }
        *o = acc;
      }
    }
  }
}

int grid_for(int64_t rows) {
  int64_t blocks = (rows + 7) / 8;                                   // 8 warps per CTA, one row per warp per trip
  const int64_t cap = static_cast<int64_t>(a4r_num_sms()) * 16;
  return static_cast<int>(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

}  // namespace

extern "C" int a4r_id_embed_fwd(const float* table, int64_t V, int64_t D, const int64_t* ids, int64_t B, int64_t S1,
                                void* emb, void* hist, a4r_stream_t stream) {
  A4R_CHECK_ARG(V >= 1 && D > 0 && D % 4 == 0 && B >= 0 && S1 >= 2, "id_embed_fwd: bad sizes (V=%lld D=%lld B=%lld S1=%lld)",
                (long long)V, (long long)D, (long long)B, (long long)S1);
  if (B == 0) return A4R_OK;
  A4R_CHECK_ARG(table && ids && emb, "id_embed_fwd: NULL pointer");
  A4R_CHECK_ARG(a4r_aligned16(table) && (reinterpret_cast<uintptr_t>(emb) & 7u) == 0 &&
                    (reinterpret_cast<uintptr_t>(hist) & 7u) == 0,
                "id_embed_fwd: table must be 16B aligned, emb / hist 8B aligned");
  int rc = a4r_device_check();
  if (rc != A4R_OK) return rc;
  IdFwdParams p;
  p.table = table, p.ids = ids, p.emb = static_cast<__nv_bfloat16*>(emb), p.hist = static_cast<__nv_bfloat16*>(hist);
  p.R = B * S1 * 2, p.S1 = S1, p.D = D, p.V = V;
  id_embed_gather_kernel<<<grid_for(p.R), 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  A4R_LAUNCH_OK();
  a4r_count_launch(1);
  return A4R_OK;
}

extern "C" int a4r_id_embed_bwd(const int64_t* sorted_ids, const int64_t* order, const void* d_emb, const void* d_hist,
                                float* grad, int64_t V, int64_t D, int64_t B, int64_t S1, int64_t padding_idx,
                                int32_t accumulate, a4r_stream_t stream) {
  A4R_CHECK_ARG(V >= 1 && D > 0 && D % 4 == 0 && B >= 0 && S1 >= 2, "id_embed_bwd: bad sizes (V=%lld D=%lld B=%lld S1=%lld)",
                (long long)V, (long long)D, (long long)B, (long long)S1);
  if (B == 0) return A4R_OK;
  A4R_CHECK_ARG(sorted_ids && order && d_emb && grad, "id_embed_bwd: NULL pointer");
  A4R_CHECK_ARG((reinterpret_cast<uintptr_t>(d_emb) & 3u) == 0 && (reinterpret_cast<uintptr_t>(d_hist) & 3u) == 0 &&
                    (reinterpret_cast<uintptr_t>(grad) & 7u) == 0,
                "id_embed_bwd: d_emb / d_hist must be 4B aligned, grad 8B aligned");
  int rc = a4r_device_check();
  if (rc != A4R_OK) return rc;
  IdBwdParams p;
  p.sorted = sorted_ids, p.order = order, p.d_emb = static_cast<const __nv_bfloat16*>(d_emb);
  p.d_hist = static_cast<const __nv_bfloat16*>(d_hist), p.grad = grad;
  p.R = B * S1 * 2, p.S1 = S1, p.D = D, p.V = V, p.skip_idx = padding_idx, p.accumulate = accumulate != 0;
  id_embed_bwd_kernel<<<grid_for(p.R), 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  A4R_LAUNCH_OK();
  a4r_count_launch(1);
  return A4R_OK;
}
