// adapter_rows_sm100.cu — K5: the Houlsby adapter block in ONE pass over the hidden states.
//
//   a   = h + W_u · act(W_d · h + b_d) + b_u            AdapterBlock.forward, Downstream/Text/model/modules.py:131-134
//   out = LayerNorm(a + input) | a + input | a          BertAdaptedSelfOutput.forward (model.py:292-297) / VITAdaptedOutput /
//                                                       VITAdaptedSelfOutput (Downstream/CV/model/model.py:182-212)
//
// TMEM hands an epilogue thread one token ROW.  Every epilogue thread keeps that layout from the accumulator to the result and
// ALL global traffic is TMA, so no staging transpose into a coalesced (row-distributed) layout is needed: measured, the
// skeleton of a staged formulation alone cost 20.6 us per 128-token tile against 13.4 us of HBM time (DESIGN.md §4.5).
//   warp 0   TMA producer of the down-projection operands (h k-blocks + W_d k-blocks, NSTAGE-deep ring);
//   warp 20  TMA producer of W_u: 4 KB chunks ([32 output columns x 64] bf16) re-streamed from L2 for every tile through a ring
//            of NWU slots.  (Resident in shared memory, W_u would take 96 KB of the 227 KB and leave room for a 2-stage operand
//            ring only — a third of the tile time was then the epilogue waiting for the NEXT tile's down-projection, 12 k-blocks
//            at two DRAM round trips in flight.  Re-reading 96 KB per tile from L2 costs 1/8 more L2->SM traffic and frees the
//            room for a 4-stage ring, a fourth residual box per group and double result boxes.)
//   warp 1   tcgen05 issuer: S1 = h · W_dᵀ, then U = s · W_uᵀ in 32-column chunks, chunk c into TMEM stage c & 1;
//   warps 2, 3  TMA producers of the RESIDUALS, one per epilogue group: [128 x 32] boxes of h and input (SWIZZLE_64B) through a
//            ring of IN_BOXES single boxes per group (each ring has ONE consumer group: no cross-group barrier phases);
//   warps 4-19 epilogue in two groups of 8 warps (chunk parity): residual rows from shared memory (conflict-free 16-byte
//            reads), z = U + b_u + h + input in registers, then
//              tail 1 / 2: bf16 row segment -> the warp's private 1 KB box -> TMA store (no barrier wider than a warp);
//              tail 0: z is parked as packed bf16 in 384 TMEM columns (tcgen05.st) while the row statistics accumulate,
//                      [training: also TMA-stored to z_out], and a second pass reads it back (tcgen05.ld), normalises
//                      and TMA-stores the result.  Nothing is re-read from L2.
// While one group computes, the other waits for / reads its operands: the phases of the two groups overlap.
#include <stdlib.h>

#include "a4r_common.cuh"

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int RP = 64;
constexpr int CC = 32;                        // columns per up-projection chunk
#ifndef A4R_K5_L2HINT
#define A4R_K5_L2HINT 1
#endif
#ifndef A4R_K5_NSTAGE          // (tuning builds only: tools/k5_variants.sh)
#define A4R_K5_NSTAGE 4
#define A4R_K5_NWU 4
#define A4R_K5_INBOXES 4
#endif
constexpr int NSTAGE = A4R_K5_NSTAGE;
constexpr int NWU = A4R_K5_NWU;               // W_u chunk ring (4 KB slots)
constexpr int WU_CHUNK = CC * 128;            // 32 rows of W_u x 64 bf16 (SW128, K-major)
constexpr int STAGE_A = BM * BK * 2;          // 16 KB of h
constexpr int STAGE_B = RP * BK * 2;          // 8 KB of W_d
constexpr int STAGE_BYTES = STAGE_A + STAGE_B;
constexpr int S_TILE = BM * RP * 2;           // 16 KB operand tile of the up-projection (also: row-statistics exchange)
constexpr int IN_HALF = BM * CC * 2;          // 8 KB: one [128 x 32] bf16 box
constexpr int OUT_STAGE = IN_HALF;          // 16 per-warp result boxes of 1 KB = two of these; every warp owns TWO boxes
constexpr int IN_BOXES = A4R_K5_INBOXES;                   // residual boxes per group: a ring of single [128 x 32] boxes (h, input, h, ...), so
                                              // a group's next chunk is in flight while it works on the current one
constexpr int EPI_WARPS = 16;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int WU_WARP = 4 + EPI_WARPS;         // warp 20: W_u chunk producer
constexpr int THREADS = 128 + EPI_THREADS + 32;
constexpr int TMEM_COLS = 512;
constexpr int U_COL = 0;                      // two 32-column U stages
constexpr int S1_COL = 64;                    // 64 columns
constexpr int Z_COL = 128;                    // 384 columns: z as packed bf16 pairs

struct RowParams {
  const float* b_down;
  const float* b_up;
  const float* gamma;
  const float* beta;
  float* mean;
  float* rstd;
  __nv_bfloat16* s_out;
  __nv_bfloat16* u_out;
  int M, H, r, lds;
  int act, tail, has_in, store_z;
  float eps;
};

A4R_DEVICE void named_bar(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
A4R_DEVICE void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
A4R_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Shared-memory loads must have RETURNED before their ring slot is handed back to the TMA producer.  `ld.shared; mbarrier.arrive`
// only orders the ISSUE of the two: the arrive can reach the barrier while the load still sits in the shared-memory queue behind
// tensor-core operand reads and TMA traffic, the producer refills the slot, and the load returns the NEXT box's bytes (measured:
// 1-3 % of the launches at M = 161,280 returned `input` of chunk c + 2 in place of `h` of chunk c for a few rows of one warp).
// A real instruction that reads one register of each load — and that ptxas may neither drop nor sink below the arrive, because it
// is a (never-taken) shared-memory store — makes the warp wait for the data first.
A4R_DEVICE void loads_returned(uint32_t scratch_saddr, uint32_t a, uint32_t b) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
      "xor.b32 t, %1, %2;\n\t"
      "setp.eq.u32 p, t, 0x9E3779B9;\n\t"
      "@p st.shared.b32 [%0], t;\n\t}" ::"r"(scratch_saddr),
      "r"(a), "r"(b)
      : "memory");
}
A4R_DEVICE void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
adapter_rows_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmWd,
                    const __grid_constant__ CUtensorMap tmWu, const __grid_constant__ CUtensorMap tmHr,
                    const __grid_constant__ CUtensorMap tmIr, const __grid_constant__ CUtensorMap tmOut,
                    const __grid_constant__ CUtensorMap tmZ, const RowParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_wu = smem;                                          // NWU x [32][64] bf16, SW128
  uint8_t* s_ring = s_wu + NWU * WU_CHUNK;
  uint8_t* s_act = s_ring + NSTAGE * STAGE_BYTES;                // [128][64] bf16, SW128
  uint8_t* s_in = s_act + S_TILE;                                // 2 groups x IN_BOXES residual boxes, SW64
  uint8_t* s_o = s_in + 2 * IN_BOXES * IN_HALF;                  // 16 x 2 x 1 KB: two result boxes per epilogue warp
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_o + 4 * OUT_STAGE);
  uint64_t* empty_bar = full_bar + NSTAGE;
  uint64_t* wu_full = empty_bar + NSTAGE;         // [NWU]
  uint64_t* wu_empty = wu_full + NWU;             // [NWU]
  uint64_t* s1_full = wu_empty + NWU;
  uint64_t* s_ready = s1_full + 1;
  uint64_t* u_full = s_ready + 1;     // [2]
  uint64_t* u_empty = u_full + 2;     // [2]
  uint64_t* in_full = u_empty + 2;                // [2][IN_BOXES]
  uint64_t* in_empty = in_full + 2 * IN_BOXES;    // [2][IN_BOXES]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_empty + 2 * IN_BOXES);
  const uint32_t scratch = smem_u32(tmem_slot + 1);   // never-read word: target of the (practically never taken) store above

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // (warp-uniform for the compiler)
  const int num_tiles = (p.M + BM - 1) / BM;
  const int nkb = p.H / BK;
  const int nch = p.H / CC;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmH);
    tma_prefetch_desc(&tmWd);
    tma_prefetch_desc(&tmWu);
    tma_prefetch_desc(&tmHr);
    tma_prefetch_desc(&tmIr);
    tma_prefetch_desc(&tmOut);
    tma_prefetch_desc(&tmZ);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < NWU; ++s) {
      mbar_init(&wu_full[s], 1);
      mbar_init(&wu_empty[s], 1);
    }
    mbar_init(s1_full, 1);
    mbar_init(s_ready, EPI_WARPS);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&u_full[s], 1);
      mbar_init(&u_empty[s], EPI_WARPS / 2);
    }
    for (int s = 0; s < 2 * IN_BOXES; ++s) {
      mbar_init(&in_full[s], 1);
      mbar_init(&in_empty[s], EPI_WARPS / 2);   // a box is consumed by ONE group of 8 warps
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
#if A4R_K5_L2HINT
  const bool saves = p.store_z != 0 || p.s_out != nullptr || p.u_out != nullptr;
  const uint64_t single_use = saves ? l2_evict_normal_policy() : l2_evict_first_policy();
#endif

  if (warp == 0) {
    // ============================== TMA producer: down-projection operands ==============================
    {                                                    // (whole warp, converged: tma_load_2d_elect)
#if A4R_K5_L2HINT
      const uint64_t keep = l2_evict_last_policy();
#endif
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          __syncwarp();
          uint8_t* sa = s_ring + stage * STAGE_BYTES;
#if A4R_K5_L2HINT
          // h is read again as the residual one tile time later (148 SMs x 0.8 MB of streams in between = the L2 capacity: half of
          // the re-reads missed): it enters L2 as evict_last, its second read and every single-use stream are evict_first
          tma_load_2d_elect_hint(&tmH, sa, &full_bar[stage], kb * BK, tile * BM, STAGE_BYTES, keep);
          tma_load_2d_elect_noarm_hint(&tmWd, sa + STAGE_A, &full_bar[stage], kb * BK, 0, keep);
#else
          tma_load_2d_elect(&tmH, sa, &full_bar[stage], kb * BK, tile * BM, STAGE_BYTES);
          tma_load_2d_elect_noarm(&tmWd, sa + STAGE_A, &full_bar[stage], kb * BK, 0);
#endif
          if (++stage == NSTAGE) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == WU_WARP) {
    // ============================== TMA producer of the W_u chunks (L2-resident: 96 KB re-streamed per tile) ==============
    {
#if A4R_K5_L2HINT
      const uint64_t keep = l2_evict_last_policy();
#endif
      uint32_t n = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int c = 0; c < nch; ++c, ++n) {
          const uint32_t slot = n % NWU;
          mbar_wait(&wu_empty[slot], ((n / NWU) & 1u) ^ 1u);
          __syncwarp();
#if A4R_K5_L2HINT
          tma_load_2d_elect_hint(&tmWu, s_wu + slot * WU_CHUNK, &wu_full[slot], 0, c * CC, WU_CHUNK, keep);
#else
          tma_load_2d_elect(&tmWu, s_wu + slot * WU_CHUNK, &wu_full[slot], 0, c * CC, WU_CHUNK);
#endif
        }
      }
    }
  } else if (warp == 2 || warp == 3) {
    // ============================== TMA producers of the residual boxes: warp 2 feeds group 0, warp 3 group 1 ==============
    // (each ring belongs to ONE group, so a consumer is never more than one phase away from its barrier)
    {
      const int g = warp - 2;
#if A4R_K5_L2HINT
      // (measured A/B, M = 161,280: evict_first on the single-use streams helps the inference variant, 191 -> 182 us, and costs the
      //  training variants 2-4 %, whose z / s stores compete for the same L2 ways: training leaves them at the default priority)
      const uint64_t drop = single_use;
#endif
      uint32_t nb = 0;                                  // running box number of this group: ring slot nb % IN_BOXES
      auto load_box = [&](const CUtensorMap* tm, int c, int tile) {
        const uint32_t b = nb % IN_BOXES;
        uint64_t* full = &in_full[g * IN_BOXES + b];
        mbar_wait(&in_empty[g * IN_BOXES + b], ((nb / IN_BOXES) & 1u) ^ 1u);
        __syncwarp();
#if A4R_K5_L2HINT
        tma_load_2d_elect_hint(tm, s_in + (g * IN_BOXES + b) * IN_HALF, full, c * CC, tile * BM, IN_HALF, drop);
#else
        tma_load_2d_elect(tm, s_in + (g * IN_BOXES + b) * IN_HALF, full, c * CC, tile * BM, IN_HALF);
#endif
        ++nb;
      };
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int c = g; c < nch; c += 2) {
          load_box(&tmHr, c, tile);
          if (p.has_in) load_box(&tmIr, c, tile);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer: the WHOLE warp, converged ==============================
    // (issued under `if (lane == 0)` every UTCHMMA sat in an ELECT / BRA.U.ANY loop — ~80 cycles per instruction on the issuing
    //  thread, 144 small MMAs per tile; see a4r_common.cuh: umma_bf16_ss_elect.  Probes are made warp-uniform by a vote.)
    {
      const uint32_t idesc_down = umma_idesc_bf16(BM, RP);
      const uint32_t idesc_up = umma_idesc_bf16(BM, CC);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t cu[2] = {0u, 0u};
      uint32_t it = 0, nwu = 0;                        // nwu: running W_u chunk number (ring slot nwu % NWU)
      auto down_kb = [&](int kb) {
        tc_fence_after();
        const uint32_t sa = smem_u32(s_ring + stage * STAGE_BYTES);
        const uint64_t adesc = umma_desc_k_sw128(sa), bdesc = umma_desc_k_sw128(sa + STAGE_A);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_bf16_ss_elect(tmem_base + S1_COL, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2), idesc_down,
                             (kb | k) != 0 ? 1u : 0u);
        umma_commit_elect(&empty_bar[stage]);
        if (++stage == NSTAGE) {
          stage = 0;
          phase ^= 1;
        }
        if (kb == nkb - 1) umma_commit_elect(s1_full);
      };
      if (static_cast<int>(blockIdx.x) < num_tiles) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          __syncwarp();
          down_kb(kb);
        }
      }
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const bool has_next = tile + static_cast<int>(gridDim.x) < num_tiles;
        mbar_wait(s_ready, it & 1);
        __syncwarp();
        tc_fence_after();
        const uint64_t adesc = umma_desc_k_sw128(smem_u32(s_act));
        int c = 0, kb = has_next ? 0 : nkb;
        while (c < nch || kb < nkb) {
          if (c < nch) {
            const int g = c & 1;
            const uint32_t slot = nwu % NWU;
            if (__all_sync(0xffffffffu, mbar_test_wait(&u_empty[g], (cu[g] & 1u) ^ 1u) && mbar_test_wait(&wu_full[slot], (nwu / NWU) & 1u))) {
              tc_fence_after();
              const uint64_t bdesc = umma_desc_k_sw128(smem_u32(s_wu + slot * WU_CHUNK));
#pragma unroll
              for (int k = 0; k < RP / 16; ++k)
                umma_bf16_ss_elect(tmem_base + U_COL + g * CC, adesc + static_cast<uint64_t>(k * 2), bdesc + static_cast<uint64_t>(k * 2),
                                   idesc_up, k != 0 ? 1u : 0u);
              umma_commit_elect(&u_full[g]);
              umma_commit_elect(&wu_empty[slot]);              // the W_u slot is free once these MMAs have read it
              ++cu[g];
              ++nwu;
              ++c;
              continue;
            }
          }
          if (kb < nkb && __all_sync(0xffffffffu, mbar_test_wait(&full_bar[stage], phase))) {
            down_kb(kb);
            ++kb;
          }
        }
      }
    }
  } else if (warp >= 4 && warp < WU_WARP) {
    // ============================== epilogue: one token row per thread, start to end ==============================
    const int ew = warp - 4;
    const int quad = warp & 3, cs = ew >> 2;             // TMEM lane quadrant; 16-column slice of S1
    const int grp = cs >> 1, hf = cs & 1;                // chunk parity this warp serves; 16-column half of the 32-column chunk
    const int rl = quad * 32 + lane;                     // row within the tile = TMEM lane
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t sact = smem_u32(s_act);
    // this thread's two 16-byte chunks inside a [128 x 32] bf16 SWIZZLE_64B box: chunk index ^ ((row >> 1) & 3)
    const uint32_t sw = static_cast<uint32_t>((rl >> 1) & 3);
    const uint32_t toff0 = rl * 64 + (((2u * hf) ^ sw) << 4), toff1 = rl * 64 + (((2u * hf + 1u) ^ sw) << 4);
    const uint32_t sin0 = smem_u32(s_in) + grp * IN_BOXES * IN_HALF;
    uint32_t nb = 0;                                     // running residual-box number of this group (as in its producer)
    const uint32_t so_w = smem_u32(s_o) + ew * 2048;     // this warp's two private out boxes (they alternate)
    uint32_t n_out = 0;
#if A4R_K5_L2HINT
    const uint64_t drop_out = single_use;
#endif
    float* stats = reinterpret_cast<float*>(s_act);      // [128][4][2] after the tile's last up-projection has retired
    uint32_t n_u = 0, it = 0;

    // Results leave per WARP: its 32 rows x 16 columns form a private 1 KB box (row pitch 32 B, no swizzle) that lane 0 hands to
    // TMA — no barrier wider than the warp, so the 16 warps drift freely instead of waiting for the slowest of a group.
    auto emit = [&](const CUtensorMap* tm, const uint32_t (&w)[8], int c, int row0) {
      const uint32_t box = so_w + (n_out & 1u) * 1024;
      ++n_out;
      __syncwarp();                                      // (elect.sync / tcgen05.* / bar.sync are .aligned: keep the warp converged)
      bulk_wait_read1_elect();                           // the store issued from THIS box two hand-overs ago has read its bytes
      __syncwarp();
      sts_v4(box + lane * 32, w[0], w[1], w[2], w[3]);
      sts_v4(box + lane * 32 + 16, w[4], w[5], w[6], w[7]);
      fence_proxy_async_smem();
      __syncwarp();
#if A4R_K5_L2HINT
      tma_store_2d_commit_elect_hint(tm, box, c * CC + hf * 16, row0 + quad * 32, drop_out);   // rows past M are clipped by the tensor map
#else
      tma_store_2d_commit_elect(tm, box, c * CC + hf * 16, row0 + quad * 32);   // rows past M are clipped by the tensor map
#endif
      __syncwarp();
    };

    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int row0 = tile * BM;
      const bool row_ok = row0 + rl < p.M;
      // ---- phase 1: s = act(S1 + b_d) -> bf16 operand tile (columns [16 cs, 16 cs + 16)) ----
      mbar_wait(s1_full, it & 1);
      __syncwarp();            // lanes may leave the spin loop in different iterations; tcgen05.ld is .aligned
      tc_fence_after();
      {
        uint32_t acc[16];
        tmem_ld_32x32b_x16(tmem_base + lane_addr + S1_COL + cs * 16, acc);
        tmem_ld_wait();
        uint32_t w[8], wu[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float pre[2], v[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int c = cs * 16 + 2 * i + e;
            pre[e] = c < p.r ? __uint_as_float(acc[2 * i + e]) + __ldg(p.b_down + c) : 0.0f;
            v[e] = c < p.r ? (p.act == 1 ? gelu_fast(pre[e]) : fmaxf(pre[e], 0.0f)) : 0.0f;
          }
          w[i] = pack_bf16x2(v[0], v[1]);
          wu[i] = pack_bf16x2(pre[0], pre[1]);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int c16 = cs * 2 + q;
          sts_v4(sact + rl * 128 + ((c16 ^ (rl & 7)) << 4), w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        }
        if (p.u_out != nullptr && row_ok) {
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int c = cs * 16 + q * 8;
            if (c < p.r)
              st_na_v4(p.u_out + static_cast<int64_t>(row0 + rl) * p.r + c,
                       make_uint4(wu[4 * q], wu[4 * q + 1], wu[4 * q + 2], wu[4 * q + 3]));
          }
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_ready);
      __syncwarp();
      if (p.s_out != nullptr) {
        // s leaves through the operand tile once every warp has written its slice: 8 lanes per 128-byte row, coalesced
        named_bar(3, EPI_THREADS);
        for (int i = threadIdx.x - 128; i < BM * 8; i += EPI_THREADS) {
          const int r_ = i >> 3, ch = i & 7;
          if (row0 + r_ < p.M && ch * 8 < p.r)
            st_na_v4(p.s_out + static_cast<int64_t>(row0 + r_) * p.lds + ch * 8, lds_v4(sact + r_ * 128 + ((ch ^ (r_ & 7)) << 4)));
          if (row0 + r_ < p.M && ch == 0 && p.lds >= p.r + 8)
            st_na_v4(p.s_out + static_cast<int64_t>(row0 + r_) * p.lds + p.r, make_uint4(0x00003F80u, 0u, 0u, 0u));
        }
      }

      // ---- pass A: z = U + b_u + h + input for this group's chunks ----
      float sum = 0.0f, sq = 0.0f;
      for (int c = grp; c < nch; c += 2) {
        uint4 h0, h1, i0 = make_uint4(0u, 0u, 0u, 0u), i1 = i0;
        {
          const uint32_t b = nb % IN_BOXES;
          mbar_wait(&in_full[grp * IN_BOXES + b], (nb / IN_BOXES) & 1u);
          h0 = lds_v4(sin0 + b * IN_HALF + toff0);
          h1 = lds_v4(sin0 + b * IN_HALF + toff1);
          loads_returned(scratch, h0.x, h1.x);
          __syncwarp();
          if (lane == 0) mbar_arrive(&in_empty[grp * IN_BOXES + b]);
          __syncwarp();
          ++nb;
        }
        if (p.has_in) {
          const uint32_t b = nb % IN_BOXES;
          mbar_wait(&in_full[grp * IN_BOXES + b], (nb / IN_BOXES) & 1u);
          i0 = lds_v4(sin0 + b * IN_HALF + toff0);
          i1 = lds_v4(sin0 + b * IN_HALF + toff1);
          loads_returned(scratch, i0.x, i1.x);
          __syncwarp();
          if (lane == 0) mbar_arrive(&in_empty[grp * IN_BOXES + b]);
          __syncwarp();
          ++nb;
        }
        mbar_wait(&u_full[grp], n_u & 1u);
        __syncwarp();
        tc_fence_after();
        uint32_t acc[16];
        tmem_ld_32x32b_x16(tmem_base + lane_addr + U_COL + grp * CC + hf * 16, acc);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&u_empty[grp]);
        __syncwarp();
        ++n_u;
        const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const uint32_t iw[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
        const float4* bu = reinterpret_cast<const float4*>(p.b_up + c * CC + hf * 16);
        uint32_t w[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 b = __ldg(bu + q);
          float2 v0 = make_float2(__uint_as_float(acc[4 * q]) + b.x, __uint_as_float(acc[4 * q + 1]) + b.y);
          float2 v1 = make_float2(__uint_as_float(acc[4 * q + 2]) + b.z, __uint_as_float(acc[4 * q + 3]) + b.w);
          v0 = __fadd2_rn(v0, bf16x2_to_f2(hw[2 * q]));
          v1 = __fadd2_rn(v1, bf16x2_to_f2(hw[2 * q + 1]));
          v0 = __fadd2_rn(v0, bf16x2_to_f2(iw[2 * q]));      // zeros without `input`
          v1 = __fadd2_rn(v1, bf16x2_to_f2(iw[2 * q + 1]));
          w[2 * q] = pack_bf16x2(v0.x, v0.y);
          w[2 * q + 1] = pack_bf16x2(v1.x, v1.y);
          // statistics of the ROUNDED row: LayerNorm's input is the bf16 tensor the backward will read
          const float2 f0 = bf16x2_to_f2(w[2 * q]), f1 = bf16x2_to_f2(w[2 * q + 1]);
          sum += (f0.x + f0.y) + (f1.x + f1.y);
          sq = fmaf(f0.x, f0.x, fmaf(f0.y, f0.y, fmaf(f1.x, f1.x, fmaf(f1.y, f1.y, sq))));
        }
        if (p.tail == 0) {
          tmem_st_32x32b_x8(tmem_base + lane_addr + Z_COL + c * (CC / 2) + hf * 8, w);
          if (p.store_z) emit(&tmZ, w, c, row0);
        } else {
          emit(&tmOut, w, c, row0);
        }
      }
      if (p.tail == 0) tmem_st_wait();
      // every up-projection of this tile has retired once both groups are here: the operand tile may be reused
      named_bar(3, EPI_THREADS);
      if (p.tail != 0) continue;

      // ---- LayerNorm: combine the four partial statistics of a row, then normalise out of the TMEM copy of z ----
      stats[(rl * 4 + cs) * 2] = sum;
      stats[(rl * 4 + cs) * 2 + 1] = sq;
      named_bar(3, EPI_THREADS);
      float s_ = 0.0f, q_ = 0.0f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        s_ += stats[(rl * 4 + k) * 2];
        q_ += stats[(rl * 4 + k) * 2 + 1];
      }
      const float inv_h = 1.0f / static_cast<float>(p.H);
      const float mu = s_ * inv_h;
      const float rs = rsqrtf(fmaxf(q_ * inv_h - mu * mu, 0.0f) + p.eps);
      if (cs == 0 && row_ok) {
        if (p.mean != nullptr) p.mean[row0 + rl] = mu;
        if (p.rstd != nullptr) p.rstd[row0 + rl] = rs;
      }
      named_bar(3, EPI_THREADS);     // the statistics have been read: phase 1 of the next tile may overwrite the operand tile
      const float2 nmu = make_float2(-mu, -mu), rs2 = make_float2(rs, rs);
      for (int c = grp; c < nch; c += 2) {
        uint32_t zw[8], w[8];
        tmem_ld_32x32b_x8(tmem_base + lane_addr + Z_COL + c * (CC / 2) + hf * 8, zw);
        const float4* gp = reinterpret_cast<const float4*>(p.gamma + c * CC + hf * 16);
        const float4* bp = reinterpret_cast<const float4*>(p.beta + c * CC + hf * 16);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 g = __ldg(gp + q), b = __ldg(bp + q);
          const float2 z0 = __fmul2_rn(__fadd2_rn(bf16x2_to_f2(zw[2 * q]), nmu), rs2);
          const float2 z1 = __fmul2_rn(__fadd2_rn(bf16x2_to_f2(zw[2 * q + 1]), nmu), rs2);
          const float2 o0 = __ffma2_rn(z0, make_float2(g.x, g.y), make_float2(b.x, b.y));
          const float2 o1 = __ffma2_rn(z1, make_float2(g.z, g.w), make_float2(b.z, b.w));
          w[2 * q] = pack_bf16x2(o0.x, o0.y);
          w[2 * q + 1] = pack_bf16x2(o1.x, o1.y);
        }
        emit(&tmOut, w, c, row0);
      }
    }
    __syncwarp();
    bulk_wait0_elect();            // the last stores have left shared memory (and are complete) before the CTA retires
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// bf16 row-major [rows, cols], leading dimension ld: box = 32 columns x 128 rows with the 64-byte swizzle (residual loads), or
// 16 columns x 32 rows unswizzled (the per-warp result boxes)
int make_tmap_box32(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, bool warp_box = false) {
  static PFN_encodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  if (fn == nullptr) return a4r_set_error(A4R_ECUDA, "cuTensorMapEncodeTiled entry point not found");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(warp_box ? 16 : CC), static_cast<cuuint32_t>(warp_box ? 32 : BM)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, warp_box ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_64B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return a4r_set_error(A4R_ECUDA, "cuTensorMapEncodeTiled (32-column box) failed (%d)", (int)r);
  return A4R_OK;
}

}  // namespace

// H <= 768: z parked as packed bf16 takes H / 2 <= 384 TMEM columns; r <= 64: the rank fits one k-block (RP)
extern "C" int a4r_adapter_ln_supported(int64_t H, int64_t r) {
  return (H % 64 == 0 && H >= 64 && H <= 768 && r % 8 == 0 && r >= 8 && r <= 64) ? 1 : 0;
}

extern "C" int a4r_adapter_ln_fwd(const a4r_adapter_args* a, a4r_stream_t stream) {
  A4R_CHECK_ARG(a != nullptr, "adapter_ln: args is NULL");
  A4R_CHECK_ARG(a->h && a->w_down && a->w_up && a->b_down && a->b_up && a->out, "adapter_ln: NULL pointer");
  A4R_CHECK_ARG(a->M >= 0 && a->M < (1ll << 31), "adapter_ln: bad M");
  A4R_CHECK_ARG(a4r_adapter_ln_supported(a->H, a->r), "adapter_ln: needs H %% 64 == 0, H <= 768, r %% 8 == 0, r <= 64 (H=%lld r=%lld)",
                (long long)a->H, (long long)a->r);
  A4R_CHECK_ARG(a->tail >= 0 && a->tail <= 2 && (a->act == 0 || a->act == 1), "adapter_ln: bad tail/act");
  A4R_CHECK_ARG(a->lds == 0 || (a->lds >= a->r && a->lds % 8 == 0 && a->lds < (1 << 20)), "adapter_ln: bad lds");
  A4R_CHECK_ARG(a->tail != 0 || (a->gamma && a->beta), "adapter_ln: tail 0 (LayerNorm) needs gamma and beta");
  A4R_CHECK_ARG(a->tail == 2 || a->input != nullptr, "adapter_ln: tails 0 and 1 add `input`");
  A4R_CHECK_ARG(a->ldh >= a->H && a->ldh % 8 == 0 && a4r_aligned16(a->h), "adapter_ln: bad h/ldh");
  A4R_CHECK_ARG(a->input == nullptr || (a->ldi >= a->H && a->ldi % 8 == 0 && a4r_aligned16(a->input)), "adapter_ln: bad input/ldi");
  A4R_CHECK_ARG(a4r_aligned16(a->w_down) && a4r_aligned16(a->w_up) && a4r_aligned16(a->out) && a4r_aligned16(a->b_up) &&
                    (a->gamma == nullptr || (a4r_aligned16(a->gamma) && a4r_aligned16(a->beta))),
                "adapter_ln: pointers must be 16B aligned");
  A4R_CHECK_ARG((a->z_out == nullptr || a4r_aligned16(a->z_out)) && (a->s_out == nullptr || a4r_aligned16(a->s_out)) &&
                    (a->u_out == nullptr || a4r_aligned16(a->u_out)),
                "adapter_ln: optional outputs must be 16B aligned");
  int rc = a4r_device_check();
  if (rc != A4R_OK) return rc;
  if (a->M == 0) return A4R_OK;

  RowParams p;
  p.b_down = a->b_down;
  p.b_up = a->b_up;
  p.gamma = a->gamma;
  p.beta = a->beta;
  p.mean = a->mean;
  p.rstd = a->rstd;
  p.s_out = static_cast<__nv_bfloat16*>(a->s_out);
  p.u_out = static_cast<__nv_bfloat16*>(a->u_out);
  p.M = static_cast<int>(a->M);
  p.H = static_cast<int>(a->H);
  p.r = static_cast<int>(a->r);
  p.lds = a->lds == 0 ? p.r : static_cast<int>(a->lds);
  p.act = a->act;
  p.tail = a->tail;
  p.has_in = (a->tail != 2 && a->input != nullptr) ? 1 : 0;
  p.store_z = (a->tail == 0 && a->z_out != nullptr) ? 1 : 0;
  p.eps = a->eps;

  CUtensorMap tmH, tmWd, tmWu, tmHr, tmIr, tmOut, tmZ;
  if ((rc = a4r_make_tmap_bf16(&tmH, a->h, a->M, a->H, a->ldh, BM)) != A4R_OK) return rc;
  if ((rc = a4r_make_tmap_bf16(&tmWd, a->w_down, a->r, a->H, a->H, RP)) != A4R_OK) return rc;
  if ((rc = a4r_make_tmap_bf16(&tmWu, a->w_up, a->H, a->r, a->r, CC)) != A4R_OK) return rc;
  if ((rc = make_tmap_box32(&tmHr, a->h, a->M, a->H, a->ldh)) != A4R_OK) return rc;
  if (p.has_in) {
    if ((rc = make_tmap_box32(&tmIr, a->input, a->M, a->H, a->ldi)) != A4R_OK) return rc;
  } else {
    tmIr = tmHr;
  }
  if ((rc = make_tmap_box32(&tmOut, a->out, a->M, a->H, a->H, true)) != A4R_OK) return rc;
  if (p.store_z) {
    if ((rc = make_tmap_box32(&tmZ, a->z_out, a->M, a->H, a->H, true)) != A4R_OK) return rc;
  } else {
    tmZ = tmOut;
  }
  const size_t smem = static_cast<size_t>(NWU) * WU_CHUNK + NSTAGE * STAGE_BYTES + S_TILE + 2 * IN_BOXES * IN_HALF + 4 * OUT_STAGE +
                      48 * sizeof(uint64_t) + 16 + 1024;
  static_assert(NWU * WU_CHUNK + NSTAGE * STAGE_BYTES + S_TILE + 2 * IN_BOXES * IN_HALF + 4 * OUT_STAGE + 48 * 8 + 16 + 1024 <= 232448,
                "shared-memory plan exceeds 227 KB");
  A4R_CUDA_OK(cudaFuncSetAttribute(adapter_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int tiles = (p.M + BM - 1) / BM;
  const int grid = tiles < a4r_num_sms() ? tiles : a4r_num_sms();
  adapter_rows_kernel<<<grid, THREADS, smem, static_cast<cudaStream_t>(stream)>>>(tmH, tmWd, tmWu, tmHr, tmIr, tmOut, tmZ, p);
  A4R_LAUNCH_OK();
  a4r_count_launch(1);
  return A4R_OK;
}
