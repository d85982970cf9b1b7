// Train-batch assembly on the device (SURVEY.md §8f-1): negative sampling + item-id -> token-row gather.
//
// Replaces BuildTrainDataset.__getitem__ (Downstream/Text/data_utils/dataset.py:24-49), which the reference runs in
// DataLoader worker processes: per user a Python rejection loop `random.randint(1, item_num)` until the draw is not in the
// user's sequence (one negative per history position, :36-40), then a NumPy fancy index `item_content[sample_items]`
// (:46) that copies 2 x (S+1) token rows of 2L int64 per user.
//
// One warp per (user, slot j in [0, S]):
//   * the lanes hold the user's left-padded sequence (slot j of every 32-wide chunk), so "is the candidate in the
//     sequence" is one compare + __any_sync per chunk;
//   * the candidate of attempt a is a pure function of (seed, offset + (user * (S+1) + j) * 64 + a) — stateless, so a
//     batch can be re-generated from its (seed, offset) and ranks need no RNG state exchange; the uniform integer in
//     [1, item_num] is the multiply-high of a 64-bit draw (bias < item_num / 2^64, Python's randint rejects instead);
//   * the negative exists only where the reference creates one: a real (non-padding) slot that is not the last (:41);
//   * the warp then copies the positive and the negative token row with 128-bit accesses (2L int64 = 30 uint4 for L = 30)
//     and lane 0 writes log_mask[b, j] = (seq[b, j] != 0) for j < S.
// HBM-bound: algorithmic bytes per user = 2(S+1) rows x 2L x 8 B read + the same written (+ ids): 40,320 B at S=20, L=30.
#include "a4r_common.cuh"

namespace {

constexpr int kMaxAttempts = 64;   // P(a draw is rejected) <= (S+1)/item_num; 64 consecutive rejections never happen
                                   // unless item_num <= S+1, where the reference's loop would not terminate either

struct SampleParams {
  const int64_t* seqs;      // [B, S1] left-padded item ids, 0 = padding
  const int64_t* content;   // [item_num + 1, W] token rows (ids | attention mask), row 0 = padding item
  const int64_t* neg_in;    // optional [B, S1]: use these negatives instead of sampling (parity tests / replay)
  int64_t* out;             // [B, S1, 2, W]
  float* log_mask;          // [B, S]
  int64_t* neg_out;         // [B, S1] the negative ids actually used
  int* fail;                // set to 1 if a slot exhausted kMaxAttempts
  int64_t B, S1, W, item_num;
  uint64_t seed, offset;
};

__global__ void __launch_bounds__(256) sample_gather_kernel(SampleParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t slots = p.B * p.S1;
  for (int64_t slot = warp; slot < slots; slot += nwarps) {
    const int64_t b = slot / p.S1, j = slot - b * p.S1;
    const int64_t* seq = p.seqs + b * p.S1;
    const int64_t pos = seq[j];
    int64_t neg = 0;
    if (p.neg_in != nullptr) {
      neg = p.neg_in[slot];
    } else if (pos != 0 && j != p.S1 - 1) {
      bool done = false;
      for (int a = 0; a < kMaxAttempts && !done; ++a) {
        const uint64_t r = rng64(p.seed, p.offset + static_cast<uint64_t>(slot) * kMaxAttempts + a);
        const int64_t cand = 1 + static_cast<int64_t>(__umul64hi(r, static_cast<uint64_t>(p.item_num)));
        bool hit = false;
        for (int64_t c0 = 0; c0 < p.S1; c0 += 32) {
          const int64_t v = (c0 + lane < p.S1) ? seq[c0 + lane] : 0;
          hit = hit || __any_sync(0xffffffffu, v == cand);
        }
        if (!hit) {
          neg = cand;
          done = true;
        }
      }
      if (!done && lane == 0) *p.fail = 1;
    }
    if (lane == 0) {
      p.neg_out[slot] = neg;
      if (j < p.S1 - 1) p.log_mask[b * (p.S1 - 1) + j] = pos != 0 ? 1.0f : 0.0f;
    }
    if (p.content == nullptr) continue;   // ids-only mode (the id item tower): the ids are seqs and neg_out themselves
    // gather: out[b, j, 0, :] = content[pos], out[b, j, 1, :] = content[neg]   (W int64 = W/2 uint4)
    const int vec = static_cast<int>(p.W >> 1);
    const uint4* src0 = reinterpret_cast<const uint4*>(p.content + pos * p.W);
    const uint4* src1 = reinterpret_cast<const uint4*>(p.content + neg * p.W);
    uint4* dst = reinterpret_cast<uint4*>(p.out + slot * 2 * p.W);
    for (int i = lane; i < 2 * vec; i += 32) {
      const uint4 v = i < vec ? __ldg(src0 + i) : __ldg(src1 + (i - vec));
      __stcs(dst + i, v);   // written once, read by the next kernel from L2/HBM: streaming store
    }
  }
}

}  // namespace

extern "C" int a4r_sample_train_batch(const int64_t* seqs, const int64_t* item_content, const int64_t* neg_in, int64_t* out,
                                      float* log_mask, int64_t* neg_out, int32_t* fail_flag, int64_t B, int64_t S1,
                                      int64_t W, int64_t item_num, uint64_t seed, uint64_t offset, a4r_stream_t stream_) {
  const bool ids_only = item_content == nullptr;
  A4R_CHECK_ARG(B >= 0 && S1 >= 2 && (ids_only ? W == 0 : (W > 0 && W % 2 == 0)) && item_num >= 1,
                "sample_train_batch: bad sizes (B=%lld S1=%lld W=%lld)", (long long)B, (long long)S1, (long long)W);
  if (B == 0) return A4R_OK;   // empty batch: the (empty) output buffers may legitimately be NULL
  A4R_CHECK_ARG(seqs && (ids_only || out) && log_mask && neg_out && fail_flag, "sample_train_batch: NULL pointer");
  A4R_CHECK_ARG(ids_only || (a4r_aligned16(item_content) && a4r_aligned16(out)),
                "sample_train_batch: item_content / out must be 16B aligned");
  int rc = a4r_device_check();
  if (rc != A4R_OK) return rc;
  SampleParams p;
  p.seqs = seqs, p.content = item_content, p.neg_in = neg_in, p.out = out, p.log_mask = log_mask, p.neg_out = neg_out;
  p.fail = fail_flag, p.B = B, p.S1 = S1, p.W = W, p.item_num = item_num, p.seed = seed, p.offset = offset;
  const int64_t slots = B * S1;
  int64_t blocks = (slots + 7) / 8;                                  // 8 warps per CTA, one slot per warp per trip
  const int64_t cap = static_cast<int64_t>(a4r_num_sms()) * 8;       // a multiple of the SM count; grid-stride beyond
  if (blocks > cap) blocks = cap;
  sample_gather_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream_)>>>(p);
  A4R_LAUNCH_OK();
  a4r_count_launch(1);
  return A4R_OK;
}
