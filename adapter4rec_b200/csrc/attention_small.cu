// attention_small.cu — K3: whole-sequence attention for short sequences (L <= 32), forward + backward.
//
// Text items have L = 30 tokens (BERT/RoBERTa, 12 heads x 64) and SASRec histories S <= 32 (2 heads x 32):
// an entire (sequence, head) problem — Q, K, V of 32 x DH — fits in 12 KB of shared memory, so ONE WARP
// owns one (sequence, head) and runs the two tiny contractions on the legacy mma.sync path.  This kernel is
// HBM-bound by construction (reads q,k,v once, writes ctx once: 4 x H x 2 B per token; SURVEY.md §8d), so
// tcgen05/TMEM would add nothing here; the tensor-pipe budget is spent in gemm_sm100.cu.
//
// Semantics follow the reference exactly:
//   scores = q·kᵀ * scale  +  mask_neg * [key masked]  +  mask_neg * [causal and j > i]      (fp32)
//   p = softmax(scores) over the L real keys;  ctx = p·v
// BERT (transformers eager path): mask_neg = finfo(float32).min, key mask from the item's attention mask
// (Downstream/Text/model/encoders.py:51-53).  SASRec: mask_neg = -1e9, causal AND key-valid
// (encoders.py:25-28, modules.py:39-42).  The mask is ADDITIVE and finite, so a fully masked query row
// degenerates to a uniform distribution over all L keys, exactly as in the reference.
#include "a4r_common.cuh"
#include "mma_sync.cuh"

namespace {

constexpr int LP = 32;            // padded sequence length
constexpr int WARPS_PER_CTA = 4;

struct AttnParams {
  const __nv_bfloat16* qkv;   // [N*L, ld_qkv]: q | k | v, each heads*DH wide
  __nv_bfloat16* out;         // fwd: ctx [N*L, ld_out];   bwd: dqkv [N*L, ld_qkv]
  const __nv_bfloat16* dout;  // bwd: dctx [N*L, ld_out]
  const void* mask;           // [N, mask_ld] int64 or f32 (non-zero = valid key) or NULL
  int64_t ld_qkv, ld_out, mask_ld;
  int N, L, heads;
  int mask_dtype;  // 0 none, 1 int64, 2 f32
  // packed (variable-length) mode: sequence n owns token rows [cu_seqlens[n], cu_seqlens[n+1]) of qkv / out / dout,
  // at most 32 of them; the key mask, if any, is then indexed by TOKEN ROW instead of [n, j].  NULL = fixed length L.
  const int32_t* cu_seqlens;
  int causal;
  float scale, mask_neg;
  uint32_t drop_thr16;  // 0 = no dropout on the attention probabilities
  float drop_scale;
  uint64_t drop_seed, drop_offset;
};

// dropout mask of the probability tile of (sequence n, head h): element (i, j), with nt = j / 8, t = (j % 8) / 2,
// e = j % 2, uses lane ((nt & 1) * 2 + e) of rng64(seed, offset + ((n*heads + h) * 32 + i) * 8 + (nt >> 1) * 4 + t),
// i.e. one 64-bit draw serves the 4 probabilities a thread owns in two adjacent n-tiles (no draw is shared or wasted).
A4R_DEVICE void prob_dropout(float (&s)[2][4][4], const AttnParams& p, int n, int h, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const uint64_t base = p.drop_offset + (static_cast<uint64_t>(n) * p.heads + h) * (32 * 8);
  const uint64_t seed = rng_seed(p.drop_seed);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int i = mt * 16 + hh * 8 + g;
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        const uint64_t r = rng64(seed, base + static_cast<uint64_t>(i) * 8 + np * 4 + t);
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            float& x = s[mt][np * 2 + q][hh * 2 + e];
            x = rng_keep(r, q * 2 + e, p.drop_thr16) ? x * p.drop_scale : 0.0f;
          }
      }
    }
}

// A tile in shared memory: ROWS x COLS bf16, row-major, 16-byte chunks XOR-swizzled by the row so that ldmatrix
// (8 rows x 16 B) is bank-conflict free.  COLS is 32, 64 or 128 (4, 8 or 16 chunks per row).
template <int COLS>
struct Tile {
  static constexpr int kChunks = COLS / 8;
  static constexpr int kBytes = LP * COLS * 2;
  A4R_DEVICE static uint32_t off(int row, int chunk) {
    // 128 B rows: xor with row; 64 B rows: two rows share a 128 B bank line, so xor with row/2.  256 B rows: xor with
    // row & 15, so 8 consecutive rows at one logical chunk land on 8 different (physical chunk & 7), i.e. bank groups.
    const int x = COLS >= 64 ? row : (row >> 1);
    return static_cast<uint32_t>(row * COLS * 2 + (((chunk ^ x) & (kChunks - 1)) << 4));
  }
};

// A-operand fragment (16 rows x 16 k) from a row-major [m][k] tile: rows m0.., k columns k0..
template <int COLS>
A4R_DEVICE void load_a(uint32_t (&a)[4], uint32_t base, int m0, int k0, int lane) {
  // matrices: (m0..+8,k0..+8) (m0+8..,k0..) (m0..,k0+8..) (m0+8..,k0+8..)
  const int mi = lane >> 3, r = lane & 7;
  const int row = m0 + r + ((mi & 1) << 3);
  const int chunk = (k0 >> 3) + (mi >> 1);
  ldsm_x4(a, base + Tile<COLS>::off(row, chunk));
}
// A-operand fragment of Xᵀ where X is stored row-major [k][m]: A[m][k] = X[k][m]
template <int COLS>
A4R_DEVICE void load_a_t(uint32_t (&a)[4], uint32_t base, int m0, int k0, int lane) {
  // matrices (trans): X[k0..+8][m0..+8], X[k0..][m0+8..], X[k0+8..][m0..], X[k0+8..][m0+8..]
  const int mi = lane >> 3, r = lane & 7;
  const int row = k0 + r + ((mi >> 1) << 3);
  const int chunk = (m0 >> 3) + (mi & 1);
  ldsm_x4_t(a, base + Tile<COLS>::off(row, chunk));
}
// B-operand fragments for TWO adjacent n-tiles (n0..n0+16) x 16 k from a tile stored [n][k] (k contiguous)
// b[0..1] -> n-tile n0, b[2..3] -> n-tile n0+8
template <int COLS>
A4R_DEVICE void load_b_nk(uint32_t (&b)[4], uint32_t base, int n0, int k0, int lane) {
  // matrices: [n0..+8][k0..+8], [n0..][k0+8..], [n0+8..][k0..], [n0+8..][k0+8..]
  const int mi = lane >> 3, r = lane & 7;
  const int row = n0 + r + ((mi >> 1) << 3);
  const int chunk = (k0 >> 3) + (mi & 1);
  ldsm_x4(b, base + Tile<COLS>::off(row, chunk));
}
// same, from a tile stored [k][n] (n contiguous): needs the transposing load
template <int COLS>
A4R_DEVICE void load_b_kn(uint32_t (&b)[4], uint32_t base, int n0, int k0, int lane) {
  // matrices (trans): [k0..+8][n0..+8], [k0+8..][n0..], [k0..][n0+8..], [k0+8..][n0+8..]
  const int mi = lane >> 3, r = lane & 7;
  const int row = k0 + r + ((mi & 1) << 3);
  const int chunk = (n0 >> 3) + (mi >> 1);
  ldsm_x4_t(b, base + Tile<COLS>::off(row, chunk));
}

// global [L rows x DH] (row stride ld) -> swizzled smem tile with 16-byte cp.async (LDGSTS: no register staging, half the
// instructions of ld + st); rows >= L are zero-filled (src-size 0).  Completion: cp_async_wait_all() + __syncwarp().
template <int DH>
A4R_DEVICE void load_tile(uint8_t* tile, const __nv_bfloat16* g, int64_t ld, int L, int lane) {
  constexpr int CH = DH / 8;
  const uint32_t base = smem_u32(tile);
#pragma unroll
  for (int i = lane; i < LP * CH; i += 32) {
    const int row = i / CH, ch = i % CH;
    const bool ok = row < L;
    const __nv_bfloat16* src = g + (ok ? static_cast<int64_t>(row) * ld + ch * 8 : 0);
    const int sz = ok ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(base + Tile<DH>::off(row, ch)), "l"(src), "r"(sz)
                 : "memory");
  }
}
A4R_DEVICE void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int DH>
A4R_DEVICE void store_tile(const uint8_t* tile, __nv_bfloat16* g, int64_t ld, int L, int lane) {
  constexpr int CH = DH / 8;
#pragma unroll
  for (int i = lane; i < LP * CH; i += 32) {
    const int row = i / CH, ch = i % CH;
    if (row < L) st_na_v4(g + static_cast<int64_t>(row) * ld + ch * 8, *reinterpret_cast<const uint4*>(tile + Tile<DH>::off(row, ch)));
  }
}
// write an accumulator tile set (2 m-tiles x NT n-tiles) as bf16 into a swizzled [32][COLS] tile
template <int COLS, int NT>
A4R_DEVICE void acc_to_tile(uint8_t* tile, const float (&acc)[2][NT][4], float s0a, float s0b, float s1a, float s1b, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const float sa = mt == 0 ? s0a : s1a, sb = mt == 0 ? s0b : s1b;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int r0 = mt * 16 + g, col = nt * 8 + 2 * t;
      *reinterpret_cast<uint32_t*>(tile + Tile<COLS>::off(r0, col >> 3) + (col & 7) * 2) =
          pack_bf16x2(acc[mt][nt][0] * sa, acc[mt][nt][1] * sa);
      *reinterpret_cast<uint32_t*>(tile + Tile<COLS>::off(r0 + 8, col >> 3) + (col & 7) * 2) =
          pack_bf16x2(acc[mt][nt][2] * sb, acc[mt][nt][3] * sb);
    }
  }
}

// where sequence n lives: first token row, its length, and the index of its first mask element
struct SeqSpan {
  int64_t row0, mask0;
  int L;
};
A4R_DEVICE SeqSpan seq_span(const AttnParams& p, int n) {
  SeqSpan s;
  if (p.cu_seqlens != nullptr) {
    const int a = __ldg(p.cu_seqlens + n), b = __ldg(p.cu_seqlens + n + 1);
    s.row0 = a, s.mask0 = a, s.L = b - a;
  } else {
    s.row0 = static_cast<int64_t>(n) * p.L, s.mask0 = static_cast<int64_t>(n) * p.mask_ld, s.L = p.L;
  }
  return s;
}
A4R_DEVICE bool key_valid(const AttnParams& p, const SeqSpan& sq, int j) {
  if (p.mask_dtype == 1) return reinterpret_cast<const int64_t*>(p.mask)[sq.mask0 + j] != 0;
  if (p.mask_dtype == 2) return reinterpret_cast<const float*>(p.mask)[sq.mask0 + j] != 0.0f;
  return true;
}

// S = Q·Kᵀ*scale + additive masks, then row softmax.  On return s[][][] holds normalised probabilities
// (columns >= L are exactly 0).  Thread (g = lane/4, t = lane%4) owns rows {g, g+8, 16+g, 24+g} and, in
// n-tile nt, columns nt*8 + 2t, +1.
template <int DH>
A4R_DEVICE void scores_softmax(float (&s)[2][4][4], uint32_t sQ, uint32_t sK, const AttnParams& p, int L, int lane,
                               uint32_t keymask_bits) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[mt][nt][e] = 0.0f;
#pragma unroll
  for (int k0 = 0; k0 < DH; k0 += 16) {
    uint32_t a0[4], a1[4];
    load_a<DH>(a0, sQ, 0, k0, lane);
    load_a<DH>(a1, sQ, 16, k0, lane);
#pragma unroll
    for (int np = 0; np < 2; ++np) {
      uint32_t b[4];
      load_b_nk<DH>(b, sK, np * 16, k0, lane);
      const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
      mma_bf16_16816(s[0][np * 2], a0, b0);
      mma_bf16_16816(s[0][np * 2 + 1], a0, b1);
      mma_bf16_16816(s[1][np * 2], a1, b0);
      mma_bf16_16816(s[1][np * 2 + 1], a1, b1);
    }
  }
  const int g = lane >> 2, t = lane & 3;
  // additive term of this thread's 8 columns, computed once per (sequence, head): -inf beyond L, mask_neg for a masked key
  float colneg[4][2];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int j = nt * 8 + 2 * t + e;
      colneg[nt][e] = j >= L ? -INFINITY : (((keymask_bits >> j) & 1u) ? 0.0f : p.mask_neg);
    }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // h=0: row g (+16mt), h=1: row g+8
      const int i = mt * 16 + h * 8 + g;
      float mx = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          float v = fmaf(s[mt][nt][h * 2 + e], p.scale, colneg[nt][e]);
          // ONE additive term whether the key is masked, in the future, or both (encoders.py:25-28)
          if (p.causal && nt * 8 + 2 * t + e > i && colneg[nt][e] == 0.0f) v += p.mask_neg;
          s[mt][nt][h * 2 + e] = v;
          mx = fmaxf(mx, v);
        }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      float sum = 0.0f;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float ex = __expf(s[mt][nt][h * 2 + e] - mx);
          s[mt][nt][h * 2 + e] = ex;
          sum += ex;
        }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      const float inv = 1.0f / sum;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) s[mt][nt][h * 2 + e] *= inv;
    }
  }
}

A4R_DEVICE uint32_t build_keymask(const AttnParams& p, const SeqSpan& sq, int lane) {
  const bool ok = lane < sq.L ? key_valid(p, sq, lane) : false;
  return __ballot_sync(0xffffffffu, ok);
}

// C-fragment pair (n-tiles 2j, 2j+1) of a 16-row m-tile -> A fragment for k-step j
A4R_DEVICE void acc_to_a(uint32_t (&a)[4], const float (&c0)[4], const float (&c1)[4]) {
  a[0] = pack_bf16x2(c0[0], c0[1]);
  a[1] = pack_bf16x2(c0[2], c0[3]);
  a[2] = pack_bf16x2(c1[0], c1[1]);
  a[3] = pack_bf16x2(c1[2], c1[3]);
}

template <int DH>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 3) attn_fwd_kernel(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t smem_attn[];
  constexpr int TB = Tile<DH>::kBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* my = smem_attn + warp * 3 * TB;
  const int64_t total = static_cast<int64_t>(p.N) * p.heads;
  for (int64_t w = static_cast<int64_t>(blockIdx.x) * WARPS_PER_CTA + warp; w < total;
       w += static_cast<int64_t>(gridDim.x) * WARPS_PER_CTA) {
    const int n = static_cast<int>(w / p.heads), h = static_cast<int>(w % p.heads);
    const int64_t Hd = static_cast<int64_t>(p.heads) * DH;
    const SeqSpan sq = seq_span(p, n);
    const __nv_bfloat16* q = p.qkv + sq.row0 * p.ld_qkv + h * DH;
    load_tile<DH>(my, q, p.ld_qkv, sq.L, lane);
    load_tile<DH>(my + TB, q + Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(my + 2 * TB, q + 2 * Hd, p.ld_qkv, sq.L, lane);
    const uint32_t km = build_keymask(p, sq, lane);
    cp_async_wait_all();
    __syncwarp();
    const uint32_t sQ = smem_u32(my), sK = sQ + TB, sV = sK + TB;
    float s[2][4][4];
    scores_softmax<DH>(s, sQ, sK, p, sq.L, lane, km);
    if (p.drop_thr16 != 0) prob_dropout(s, p, n, h, lane);  // dropout on the probabilities (train mode)
    // O = P·V
    float o[2][DH / 8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) o[mt][nt][e] = 0.0f;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t a0[4], a1[4];
      acc_to_a(a0, s[0][2 * ks], s[0][2 * ks + 1]);
      acc_to_a(a1, s[1][2 * ks], s[1][2 * ks + 1]);
#pragma unroll
      for (int np = 0; np < DH / 16; ++np) {
        uint32_t b[4];
        load_b_kn<DH>(b, sV, np * 16, ks * 16, lane);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16_16816(o[0][np * 2], a0, b0);
        mma_bf16_16816(o[0][np * 2 + 1], a0, b1);
        mma_bf16_16816(o[1][np * 2], a1, b0);
        mma_bf16_16816(o[1][np * 2 + 1], a1, b1);
      }
    }
    __syncwarp();
    acc_to_tile<DH, DH / 8>(my, o, 1.f, 1.f, 1.f, 1.f, lane);  // reuse the Q tile as the staging buffer
    __syncwarp();
    store_tile<DH>(my, p.out + sq.row0 * p.ld_out + h * DH, p.ld_out, sq.L, lane);
    __syncwarp();
  }
}

// Backward: recompute P, then dV = Pᵀ·dO, dP = dO·Vᵀ, dS = P ⊙ (dP − rowsum(P ⊙ dP)) * scale,
// dQ = dS·K, dK = dSᵀ·Q.  Writes dq | dk | dv in the layout of qkv.
template <int DH>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) attn_bwd_kernel(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t smem_attn[];
  constexpr int TB = Tile<DH>::kBytes;
  constexpr int PB = Tile<32>::kBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* my = smem_attn + warp * (4 * TB + 2 * PB);
  const int64_t total = static_cast<int64_t>(p.N) * p.heads;
  for (int64_t w = static_cast<int64_t>(blockIdx.x) * WARPS_PER_CTA + warp; w < total;
       w += static_cast<int64_t>(gridDim.x) * WARPS_PER_CTA) {
    const int n = static_cast<int>(w / p.heads), h = static_cast<int>(w % p.heads);
    const int64_t Hd = static_cast<int64_t>(p.heads) * DH;
    const SeqSpan sq = seq_span(p, n);
    const __nv_bfloat16* q = p.qkv + sq.row0 * p.ld_qkv + h * DH;
    uint8_t *tQ = my, *tK = my + TB, *tV = my + 2 * TB, *tdO = my + 3 * TB, *tP = my + 4 * TB, *tdS = tP + PB;
    load_tile<DH>(tQ, q, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tK, q + Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tV, q + 2 * Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tdO, p.dout + sq.row0 * p.ld_out + h * DH, p.ld_out, sq.L, lane);
    const uint32_t km = build_keymask(p, sq, lane);
    cp_async_wait_all();
    __syncwarp();
    const uint32_t sQ = smem_u32(tQ), sK = smem_u32(tK), sV = smem_u32(tV), sdO = smem_u32(tdO), sP = smem_u32(tP),
                   sdS = smem_u32(tdS);
    float s[2][4][4];
    scores_softmax<DH>(s, sQ, sK, p, sq.L, lane, km);
    // dP = dO·Vᵀ   (B operand: V stored [key][dim] = [n][k])
    float dp[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dp[mt][nt][e] = 0.0f;
#pragma unroll
    for (int k0 = 0; k0 < DH; k0 += 16) {
      uint32_t a0[4], a1[4];
      load_a<DH>(a0, sdO, 0, k0, lane);
      load_a<DH>(a1, sdO, 16, k0, lane);
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        uint32_t b[4];
        load_b_nk<DH>(b, sV, np * 16, k0, lane);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16_16816(dp[0][np * 2], a0, b0);
        mma_bf16_16816(dp[0][np * 2 + 1], a0, b1);
        mma_bf16_16816(dp[1][np * 2], a1, b0);
        mma_bf16_16816(dp[1][np * 2 + 1], a1, b1);
      }
    }
    // with probability dropout O = (P ⊙ m)·V: dP picks up the mask, dV uses the dropped probabilities
    float sd[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) sd[mt][nt][e] = s[mt][nt][e];
    if (p.drop_thr16 != 0) {
      prob_dropout(sd, p, n, h, lane);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 4; ++e) dp[mt][nt][e] = (sd[mt][nt][e] != 0.0f) ? dp[mt][nt][e] * p.drop_scale : 0.0f;
    }
    // dS = P ⊙ (dP − δ) * scale,  δ_i = Σ_j P_ij dP_ij
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float d = 0.0f;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) d += s[mt][nt][hh * 2 + e] * dp[mt][nt][hh * 2 + e];
        d += __shfl_xor_sync(0xffffffffu, d, 1);
        d += __shfl_xor_sync(0xffffffffu, d, 2);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            dp[mt][nt][hh * 2 + e] = s[mt][nt][hh * 2 + e] * (dp[mt][nt][hh * 2 + e] - d) * p.scale;
      }
    // stage P and dS (bf16, [query][key]) for the transposed products
    acc_to_tile<32, 4>(tP, sd, 1.f, 1.f, 1.f, 1.f, lane);
    acc_to_tile<32, 4>(tdS, dp, 1.f, 1.f, 1.f, 1.f, lane);
    __syncwarp();
    // dQ = dS·K   (A from registers, B: K stored [key][dim] = [k][n])
    float acc[2][DH / 8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.0f;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t a0[4], a1[4];
      acc_to_a(a0, dp[0][2 * ks], dp[0][2 * ks + 1]);
      acc_to_a(a1, dp[1][2 * ks], dp[1][2 * ks + 1]);
#pragma unroll
      for (int np = 0; np < DH / 16; ++np) {
        uint32_t b[4];
        load_b_kn<DH>(b, sK, np * 16, ks * 16, lane);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16_16816(acc[0][np * 2], a0, b0);
        mma_bf16_16816(acc[0][np * 2 + 1], a0, b1);
        mma_bf16_16816(acc[1][np * 2], a1, b0);
        mma_bf16_16816(acc[1][np * 2 + 1], a1, b1);
      }
    }
    // dK = dSᵀ·Q and dV = Pᵀ·dO need Q and dO as [k][n] B operands and dSᵀ/Pᵀ as transposed A operands;
    // compute both before any input tile is overwritten.
    float dk[2][DH / 8][4], dv[2][DH / 8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dk[mt][nt][e] = dv[mt][nt][e] = 0.0f;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {  // k = query index
      uint32_t a0[4], a1[4], p0[4], p1[4];
      load_a_t<32>(a0, sdS, 0, ks * 16, lane);
      load_a_t<32>(a1, sdS, 16, ks * 16, lane);
      load_a_t<32>(p0, sP, 0, ks * 16, lane);
      load_a_t<32>(p1, sP, 16, ks * 16, lane);
#pragma unroll
      for (int np = 0; np < DH / 16; ++np) {
        uint32_t b[4];
        load_b_kn<DH>(b, sQ, np * 16, ks * 16, lane);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16_16816(dk[0][np * 2], a0, b0);
        mma_bf16_16816(dk[0][np * 2 + 1], a0, b1);
        mma_bf16_16816(dk[1][np * 2], a1, b0);
        mma_bf16_16816(dk[1][np * 2 + 1], a1, b1);
        uint32_t c[4];
        load_b_kn<DH>(c, sdO, np * 16, ks * 16, lane);
        const uint32_t c0[2] = {c[0], c[1]}, c1[2] = {c[2], c[3]};
        mma_bf16_16816(dv[0][np * 2], p0, c0);
        mma_bf16_16816(dv[0][np * 2 + 1], p0, c1);
        mma_bf16_16816(dv[1][np * 2], p1, c0);
        mma_bf16_16816(dv[1][np * 2 + 1], p1, c1);
      }
    }
    __syncwarp();
    acc_to_tile<DH, DH / 8>(tQ, acc, 1.f, 1.f, 1.f, 1.f, lane);
    acc_to_tile<DH, DH / 8>(tK, dk, 1.f, 1.f, 1.f, 1.f, lane);
    acc_to_tile<DH, DH / 8>(tV, dv, 1.f, 1.f, 1.f, 1.f, lane);
    __syncwarp();
    __nv_bfloat16* dq = p.out + sq.row0 * p.ld_qkv + h * DH;
    store_tile<DH>(tQ, dq, p.ld_qkv, sq.L, lane);
    store_tile<DH>(tK, dq + Hd, p.ld_qkv, sq.L, lane);
    store_tile<DH>(tV, dq + 2 * Hd, p.ld_qkv, sq.L, lane);
    __syncwarp();
  }
}

// ---- head_dim 128 ------------------------------------------------------------------------------------------------
// Scores, P and dS reduce over the head dimension and are computed once over all 128 columns, as above.  The output
// contractions (ctx = P·V; dQ = dS·K, dK = dSᵀ·Q, dV = Pᵀ·dO) run in 64-column halves, one product at a time, and
// each half is written to shared memory before the next starts, so one 2 x 8 x 4 fp32 accumulator is live instead of
// three 2 x 16 x 4 ones.  Each half overwrites the half of the input tile its product consumed, so no staging tile is
// added.  A warp stages 24 KB (forward: Q, K, V) or 36 KB (backward: Q, K, V, dO, P, dS); 2-warp CTAs let 4 forward or
// 3 backward CTAs share an SM.
constexpr int WARPS_128 = 2;

// A fragments [k-step][m-tile] of a 32 x 32 bf16 operand staged as a [32][32] tile: A = X (TRANS false) or Xᵀ (true)
template <bool TRANS>
A4R_DEVICE void load_a32(uint32_t (&a)[2][2][4], uint32_t sX, int lane) {
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      if constexpr (TRANS)
        load_a_t<32>(a[ks][mt], sX, mt * 16, ks * 16, lane);
      else
        load_a<32>(a[ks][mt], sX, mt * 16, ks * 16, lane);
    }
}

// acc = A·B[:, c0 .. c0+64): A is 32 x 32 (fragments [k-step][m-tile]), B a [k][n] tile of 128 columns
A4R_DEVICE void mma_half(float (&acc)[2][8][4], const uint32_t (&a)[2][2][4], uint32_t sB, int c0, int lane) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.0f;
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t b[4];
      load_b_kn<128>(b, sB, c0 + np * 16, ks * 16, lane);
      const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
      mma_bf16_16816(acc[0][np * 2], a[ks][0], b0);
      mma_bf16_16816(acc[0][np * 2 + 1], a[ks][0], b1);
      mma_bf16_16816(acc[1][np * 2], a[ks][1], b0);
      mma_bf16_16816(acc[1][np * 2 + 1], a[ks][1], b1);
    }
}

// bf16 of a 32 x 64 accumulator into columns c0 .. c0+64 of a swizzled [32][128] tile
A4R_DEVICE void half_to_tile(uint8_t* tile, const float (&acc)[2][8][4], int c0, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int r0 = mt * 16 + g, col = c0 + nt * 8 + 2 * t;
      *reinterpret_cast<uint32_t*>(tile + Tile<128>::off(r0, col >> 3) + (col & 7) * 2) =
          pack_bf16x2(acc[mt][nt][0], acc[mt][nt][1]);
      *reinterpret_cast<uint32_t*>(tile + Tile<128>::off(r0 + 8, col >> 3) + (col & 7) * 2) =
          pack_bf16x2(acc[mt][nt][2], acc[mt][nt][3]);
    }
}

// tile[:, c0 .. c0+64) = A·tile[:, c0 .. c0+64): the product reads only that half of B, then overwrites it
A4R_DEVICE void product_half_inplace(const uint32_t (&a)[2][2][4], uint8_t* tile, int c0, int lane) {
  float acc[2][8][4];
  mma_half(acc, a, smem_u32(tile), c0, lane);
  __syncwarp();
  half_to_tile(tile, acc, c0, lane);
}

template <>
__global__ void __launch_bounds__(WARPS_128 * 32) attn_fwd_kernel<128>(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t smem_attn[];
  constexpr int DH = 128, TB = Tile<DH>::kBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* my = smem_attn + warp * 3 * TB;
  const int64_t total = static_cast<int64_t>(p.N) * p.heads;
  for (int64_t w = static_cast<int64_t>(blockIdx.x) * WARPS_128 + warp; w < total;
       w += static_cast<int64_t>(gridDim.x) * WARPS_128) {
    const int n = static_cast<int>(w / p.heads), h = static_cast<int>(w % p.heads);
    const int64_t Hd = static_cast<int64_t>(p.heads) * DH;
    const SeqSpan sq = seq_span(p, n);
    const __nv_bfloat16* q = p.qkv + sq.row0 * p.ld_qkv + h * DH;
    uint8_t *tQ = my, *tV = my + 2 * TB;
    load_tile<DH>(tQ, q, p.ld_qkv, sq.L, lane);
    load_tile<DH>(my + TB, q + Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tV, q + 2 * Hd, p.ld_qkv, sq.L, lane);
    const uint32_t km = build_keymask(p, sq, lane);
    cp_async_wait_all();
    __syncwarp();
    float s[2][4][4];
    scores_softmax<DH>(s, smem_u32(tQ), smem_u32(my + TB), p, sq.L, lane, km);
    if (p.drop_thr16 != 0) prob_dropout(s, p, n, h, lane);
    uint32_t pa[2][2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) acc_to_a(pa[ks][mt], s[mt][2 * ks], s[mt][2 * ks + 1]);
    // O = P·V, one half at a time, staged in place of the V half it consumed
#pragma unroll 1
    for (int c0 = 0; c0 < DH; c0 += 64) product_half_inplace(pa, tV, c0, lane);
    __syncwarp();
    store_tile<DH>(tV, p.out + sq.row0 * p.ld_out + h * DH, p.ld_out, sq.L, lane);
    __syncwarp();
  }
}

template <>
__global__ void __launch_bounds__(WARPS_128 * 32) attn_bwd_kernel<128>(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t smem_attn[];
  constexpr int DH = 128, TB = Tile<DH>::kBytes, PB = Tile<32>::kBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* my = smem_attn + warp * (4 * TB + 2 * PB);
  const int64_t total = static_cast<int64_t>(p.N) * p.heads;
  for (int64_t w = static_cast<int64_t>(blockIdx.x) * WARPS_128 + warp; w < total;
       w += static_cast<int64_t>(gridDim.x) * WARPS_128) {
    const int n = static_cast<int>(w / p.heads), h = static_cast<int>(w % p.heads);
    const int64_t Hd = static_cast<int64_t>(p.heads) * DH;
    const SeqSpan sq = seq_span(p, n);
    const __nv_bfloat16* q = p.qkv + sq.row0 * p.ld_qkv + h * DH;
    uint8_t *tQ = my, *tK = my + TB, *tV = my + 2 * TB, *tdO = my + 3 * TB, *tP = my + 4 * TB, *tdS = tP + PB;
    load_tile<DH>(tQ, q, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tK, q + Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tV, q + 2 * Hd, p.ld_qkv, sq.L, lane);
    load_tile<DH>(tdO, p.dout + sq.row0 * p.ld_out + h * DH, p.ld_out, sq.L, lane);
    const uint32_t km = build_keymask(p, sq, lane);
    cp_async_wait_all();
    __syncwarp();
    const uint32_t sdO = smem_u32(tdO), sP = smem_u32(tP), sdS = smem_u32(tdS);
    float s[2][4][4];
    scores_softmax<DH>(s, smem_u32(tQ), smem_u32(tK), p, sq.L, lane, km);
    // dP = dO·Vᵀ over all 128 columns
    float dp[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dp[mt][nt][e] = 0.0f;
#pragma unroll
    for (int k0 = 0; k0 < DH; k0 += 16) {
      uint32_t a0[4], a1[4];
      load_a<DH>(a0, sdO, 0, k0, lane);
      load_a<DH>(a1, sdO, 16, k0, lane);
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        uint32_t b[4];
        load_b_nk<DH>(b, smem_u32(tV), np * 16, k0, lane);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16_16816(dp[0][np * 2], a0, b0);
        mma_bf16_16816(dp[0][np * 2 + 1], a0, b1);
        mma_bf16_16816(dp[1][np * 2], a1, b0);
        mma_bf16_16816(dp[1][np * 2 + 1], a1, b1);
      }
    }
    // dropout and dS exactly as in the 32 / 64 kernel
    float sd[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) sd[mt][nt][e] = s[mt][nt][e];
    if (p.drop_thr16 != 0) {
      prob_dropout(sd, p, n, h, lane);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 4; ++e) dp[mt][nt][e] = (sd[mt][nt][e] != 0.0f) ? dp[mt][nt][e] * p.drop_scale : 0.0f;
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float d = 0.0f;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) d += s[mt][nt][hh * 2 + e] * dp[mt][nt][hh * 2 + e];
        d += __shfl_xor_sync(0xffffffffu, d, 1);
        d += __shfl_xor_sync(0xffffffffu, d, 2);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            dp[mt][nt][hh * 2 + e] = s[mt][nt][hh * 2 + e] * (dp[mt][nt][hh * 2 + e] - d) * p.scale;
      }
    acc_to_tile<32, 4>(tP, sd, 1.f, 1.f, 1.f, 1.f, lane);
    acc_to_tile<32, 4>(tdS, dp, 1.f, 1.f, 1.f, 1.f, lane);
    __syncwarp();
    // V is no longer needed.  Each half of dQ = dS·K, dK = dSᵀ·Q, dV = Pᵀ·dO replaces the half of K, Q, dO it read.
    // The A operands come back from the staged bf16 tiles: the same values the 32 / 64 kernel packs from registers.
#pragma unroll 1
    for (int c0 = 0; c0 < DH; c0 += 64) {
      uint32_t a[2][2][4];
      load_a32<false>(a, sdS, lane);
      product_half_inplace(a, tK, c0, lane);
      load_a32<true>(a, sdS, lane);
      product_half_inplace(a, tQ, c0, lane);
      load_a32<true>(a, sP, lane);
      product_half_inplace(a, tdO, c0, lane);
    }
    __syncwarp();
    __nv_bfloat16* dq = p.out + sq.row0 * p.ld_qkv + h * DH;
    store_tile<DH>(tK, dq, p.ld_qkv, sq.L, lane);
    store_tile<DH>(tQ, dq + Hd, p.ld_qkv, sq.L, lane);
    store_tile<DH>(tdO, dq + 2 * Hd, p.ld_qkv, sq.L, lane);
    __syncwarp();
  }
}

int check_common(const a4r_attn_args* a) {
  A4R_CHECK_ARG(a != nullptr, "attention: args is NULL");
  A4R_CHECK_ARG(a->qkv && a->out, "attention: qkv/out must be non-NULL");
  A4R_CHECK_ARG(a->L >= 1 && a->L <= LP, "attention_small: L must be in [1,32] (got %lld)", (long long)a->L);
  A4R_CHECK_ARG(a->head_dim == 32 || a->head_dim == 64 || a->head_dim == 128,
                "attention_small: head_dim must be 32, 64 or 128 (got %lld)", (long long)a->head_dim);
  A4R_CHECK_ARG(a->heads >= 1 && a->N >= 0, "attention: bad heads/N");
  A4R_CHECK_ARG(a->ld_qkv >= 3 * a->heads * a->head_dim && a->ld_qkv % 8 == 0, "attention: bad ld_qkv");
  A4R_CHECK_ARG(a->ld_out >= a->heads * a->head_dim && a->ld_out % 8 == 0, "attention: bad ld_out");
  A4R_CHECK_ARG(a4r_aligned16(a->qkv) && a4r_aligned16(a->out), "attention: pointers must be 16B aligned");
  A4R_CHECK_ARG(a->mask_dtype >= 0 && a->mask_dtype <= 2, "attention: mask_dtype must be 0,1,2");
  if (a->mask_dtype != 0)
    A4R_CHECK_ARG(a->mask != nullptr && (a->cu_seqlens != nullptr || a->mask_ld >= a->L), "attention: bad mask/mask_ld");
  A4R_CHECK_ARG(a->dropout_p >= 0.0f && a->dropout_p < 1.0f, "attention: dropout_p must be in [0,1)");
  return a4r_device_check();
}

AttnParams to_params(const a4r_attn_args* a) {
  AttnParams p;
  p.qkv = static_cast<const __nv_bfloat16*>(a->qkv);
  p.out = static_cast<__nv_bfloat16*>(a->out);
  p.dout = static_cast<const __nv_bfloat16*>(a->dout);
  p.mask = a->mask;
  p.ld_qkv = a->ld_qkv;
  p.ld_out = a->ld_out;
  p.mask_ld = a->mask_ld;
  p.N = static_cast<int>(a->N);
  p.L = static_cast<int>(a->L);
  p.cu_seqlens = a->cu_seqlens;
  p.heads = static_cast<int>(a->heads);
  p.mask_dtype = a->mask_dtype;
  p.causal = a->causal;
  p.scale = a->scale;
  p.mask_neg = a->mask_neg;
  p.drop_thr16 = static_cast<uint32_t>(a->dropout_p * 65536.0f + 0.5f);
  p.drop_scale = 65536.0f / static_cast<float>(65536u - p.drop_thr16);
  p.drop_seed = a->dropout_seed;
  p.drop_offset = a->dropout_offset;
  return p;
}

// warps: warps per CTA.  per_sm: NULL caps the grid at 8 CTAs per SM; otherwise the resident CTAs per SM, found with the
// occupancy calculator when the attribute is set, so that every warp of the grid-stride loop runs the same share.
template <typename K>
int launch(K kernel, int smem, const AttnParams& p, cudaStream_t stream, bool* attr_done, int warps = WARPS_PER_CTA,
           int* per_sm = nullptr) {
  if (!*attr_done) {
    A4R_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (per_sm != nullptr) {
      A4R_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kernel, warps * 32, smem));
      if (*per_sm < 1) *per_sm = 1;
    }
    *attr_done = true;
  }
  const int64_t total = static_cast<int64_t>(p.N) * p.heads;
  int64_t blocks = (total + warps - 1) / warps;
  const int64_t cap = static_cast<int64_t>(a4r_num_sms()) * (per_sm != nullptr ? *per_sm : 8);
  if (blocks > cap) blocks = cap;
  kernel<<<static_cast<int>(blocks), warps * 32, smem, stream>>>(p);
  A4R_LAUNCH_OK();
  a4r_count_launch(1);
  return A4R_OK;
}

}  // namespace

extern "C" int a4r_attn_small_fwd(const a4r_attn_args* a, a4r_stream_t stream) {
  int rc = check_common(a);
  if (rc != A4R_OK) return rc;
  if (a->N == 0) return A4R_OK;
  const AttnParams p = to_params(a);
  static bool done64 = false, done32 = false, done128 = false;
  static int per_sm128 = 0;
  if (a->head_dim == 128)
    return launch(attn_fwd_kernel<128>, WARPS_128 * 3 * Tile<128>::kBytes, p, static_cast<cudaStream_t>(stream), &done128,
                  WARPS_128, &per_sm128);
  if (a->head_dim == 64)
    return launch(attn_fwd_kernel<64>, WARPS_PER_CTA * 3 * Tile<64>::kBytes, p, static_cast<cudaStream_t>(stream), &done64);
  return launch(attn_fwd_kernel<32>, WARPS_PER_CTA * 3 * Tile<32>::kBytes, p, static_cast<cudaStream_t>(stream), &done32);
}

extern "C" int a4r_attn_small_bwd(const a4r_attn_args* a, a4r_stream_t stream) {
  int rc = check_common(a);
  if (rc != A4R_OK) return rc;
  A4R_CHECK_ARG(a->dout != nullptr && a4r_aligned16(a->dout), "attention bwd: dout missing or unaligned");
  if (a->N == 0) return A4R_OK;
  const AttnParams p = to_params(a);
  static bool done64 = false, done32 = false, done128 = false;
  static int per_sm128 = 0;
  if (a->head_dim == 128)
    return launch(attn_bwd_kernel<128>, WARPS_128 * (4 * Tile<128>::kBytes + 2 * Tile<32>::kBytes), p,
                  static_cast<cudaStream_t>(stream), &done128, WARPS_128, &per_sm128);
  if (a->head_dim == 64)
    return launch(attn_bwd_kernel<64>, WARPS_PER_CTA * (4 * Tile<64>::kBytes + 2 * Tile<32>::kBytes), p,
                  static_cast<cudaStream_t>(stream), &done64);
  return launch(attn_bwd_kernel<32>, WARPS_PER_CTA * (4 * Tile<32>::kBytes + 2 * Tile<32>::kBytes), p,
                static_cast<cudaStream_t>(stream), &done32);
}
