// tcgen05 GEMM / implicit-GEMM convolution for sm_100a.
//
//   out[M, N] = epilogue( A[M, K] * W[N, K]^T )           fp16 operands, fp32 accumulation in TMEM
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier full/empty)
//   warp 1      MMA issuer    (tcgen05.mma, M=128, N=BN, K=16; accumulators double-buffered in TMEM)
//   warps 2..9  epilogue      (tcgen05.ld -> +bias, +residual | GEGLU -> fp16 -> swizzled smem box -> TMA store), overlaps
//               the next tile's mainloop; two warps per TMEM lane quarter, each taking every other 32-column chunk
// Template variants (chosen per problem by pick_bn / pick_cg / pick_wide):
//   CG = 2      the CTAs of a 2-CTA cluster take two vertically adjacent 128-row tiles; ONE tcgen05.mma cta_group::2 (M=256)
//               issued by the leader consumes a B tile of which each CTA staged half
//   NACC = 2    "wide" tile on top of CG = 2: one staged A tile feeds two N=BN accumulators (256 x 2BN outputs per pair),
//               three TMEM slots in rotation. The kernel is bound by the SM's shared-memory port (operand reads + TMA
//               writes), not by the tensor pipe: DESIGN.md section 4.
//
// The A operand is fetched by TMA in one of three addressing modes, so that linear layers, 1x1 convs, 3x3 convs
// (stride 1 and 2, zero padding via TMA out-of-bounds fill) and channel-concatenated inputs (two K sources) share
// one mainloop and no im2col / concat buffer is ever materialised:
//   A_GEMM      2-D map [M, K]            (optionally a second map: K = K1 ++ K2)
//   A_CONV_S1   4-D map (C, W, H, Nf)     box {64, bw, bh, bn}, tap (ky,kx) -> coordinate shift (kx-1, ky-1)
//   A_CONV_S2   5-D map (2C, W/2, 2, H/2, Nf) (even/odd pixel phases split out), box {64, bw, 1, bh, bn}
//
// Replaces, for the hot path: cuDNN/cuBLAS calls behind InflatedConv3d (reference src/models/resnet.py:10-18),
// nn.Linear / 1x1 nn.Conv2d in Transformer3DModel (src/models/transformer_3d.py:64-66,93-95), diffusers Attention
// to_q/k/v/out and FeedForward(GEGLU) (src/models/attention.py:323-361, src/models/motion_module.py:122,144,233).
#include <stdio.h>
#include <stdlib.h>

#include "ap_host.h"
#include "ap_ptx.cuh"

namespace ap {

enum { A_GEMM = 0, A_CONV_S1 = 1, A_CONV_S2 = 2 };
enum { EPI_LINEAR = 0, EPI_GEGLU = 1, EPI_GELU = 2 };   // EPI_GELU: out = gelu_erf(acc + bias), no residual / statistics

struct GemmParams {
  int M, N;                // output rows; weight rows (N % BN == 0)
  int num_m_tiles, num_n_tiles, num_kb;
  int a_mode;
  int kb_src1, kb_src2;    // 64-wide k-blocks per tap taken from source 1 / source 2
  // conv geometry (output grid) and tile box
  int Nf, Ho, Wo;
  int bw, bh, bn;
  int tiles_x, tiles_y;
  int C1;                  // channels of source 1 (A_CONV_S2 merged (phase, channel) coordinate)
  // epilogue
  const float* bias;       // [groups, Nout] fp32 or null
  int bias_group_rows;     // rows sharing one bias row (>= M -> single row)
  long long bias_ld;       // floats between bias rows (N unless several ops share one table)
  const __half* residual;  // [M, ldr] or null
  int ldr;
  __half* out;             // [M, ldo]
  int ldo;
  int n_valid;             // columns >= n_valid are not stored
  int out_f32;             // store fp32 instead of fp16 (small bias-table GEMMs)
  // TMA epilogue (per-warp 32-row x 32-column boxes staged in 64B-swizzled shared memory)
  int tma_epi;             // 1: outputs leave through TMA stores, the residual arrives through TMA loads
  int sub_w, sub_h, sub_n; // conv modes: geometry of a warp's 32-row sub-box
  int epi_double;          // double-buffered output staging when there is no residual (AP_GEMM_EPI_DOUBLE=0 disables: A/B)
  int debug;               // AP_GEMM_DEBUG: 1 = skip TMA loads (MMA pace), 2 = skip MMAs (TMA pace), 3 / 4 = skip every other
                           // B / A load (traffic sensitivity); results are garbage
  // ---- statistics fused into the epilogue (TMA epilogue only) --------------------------------------------------------
  // Producer side. Both are computed from the fp16-ROUNDED outputs (what the consumer will read) and written as per-warp
  // partials in a fixed layout: no atomics, the consumer adds them in a fixed order (bit-reproducible).
  float2* row_stat_out;    // LayerNorm of the NEXT op: {sum, sum of squares} of output row m over the columns this epilogue
                           // warp handled: [part][row_stat_ld], part = 2 * (n-group of the work item) + (warp's column half)
  long long row_stat_ld;
  float2* col_stat_out;    // GroupNorm of the NEXT op: {sum, sumsq} per output column over the 32 rows of the warp's TMEM lane
                           // quarter: [4 * m_tile + quarter][col_stat_ld]
  long long col_stat_ld;
  // Consumer side (LayerNorm folded into this GEMM): A = [x | -mean (hi, lo, hi)], W = [W diag(gamma) | colsum (hi, hi, lo)],
  // so the accumulator already holds x.W'^T - mean colsum(W') (the mean term rides on one extra k-block of the tensor
  // core; the two-source A path existed for the skip concat); the epilogue only scales by the row's rstd:
  //   out = rstd * acc + (beta.W^T + b)   [the last term arrives as `bias`]: one FMA where the bias add used to be.
  const float* ln_rstd;    // [M] fp32, written by ln_finalize_kernel from the producer's row partials
};

// NACC = 2 ("wide" tile, cta_group::2 only): one staged A tile feeds TWO N = BN accumulators (two adjacent BN-wide weight
// slabs), i.e. a 256 x 2BN output tile per CTA pair. Per 64-wide k-block and CTA the shared-memory port then moves
// A 16 KB in + 2 x 16 KB out, B 20 KB in + 20 KB out = 88 KB per 640 MMA clocks instead of 2 x 52 KB (BN = 160), which is
// what bounds the narrow tile (DESIGN.md section 4). TMEM holds three BN-wide accumulator slots used in rotation (tile i:
// slots 2i % 3 and (2i+1) % 3), so the epilogue of tile i still overlaps the mainloop of tile i+1 except for the drain
// of its first slot.
template <int BN, int CG = 1, int NACC = 1>
struct GemmCfg {
  static constexpr int BM = 128;
  static constexpr int BK = 64;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_SLAB = (BN / CG) * BK * 2;    // cta_group::2: each CTA of the pair stages half of a B slab
  static constexpr int B_BYTES = NACC * B_SLAB;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_STAGING = 8 * 4096;  // 8 epilogue warps x (2 KB output box + 2 KB residual box)
  static constexpr int MAX_SMEM = 227 * 1024 - 2048 - EPI_STAGING;
  static constexpr int STAGES_RAW = MAX_SMEM / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int ACC_SLOTS = NACC == 2 ? 3 : 2;
  static constexpr int ACC_COLS = ACC_SLOTS * BN;
  static constexpr int TMEM_COLS = (ACC_COLS <= 32) ? 32 : (ACC_COLS <= 64) ? 64 : (ACC_COLS <= 128) ? 128 : (ACC_COLS <= 256) ? 256 : 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_STAGING + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(ACC_COLS <= 512, "the accumulator slots must fit TMEM");
  static_assert(NACC == 1 || CG == 2, "wide tiles are built on cta_group::2");
  static_assert(B_SLAB % 1024 == 0, "B stage must keep 1024B alignment");
};

// erf-GELU with ONE MUFU op: erfc(z) = 2^-q(z), q(z) = z * P6(z) fitted to -log2(erfc z) on [0, 4.3] (max relative error of
// erfc 4.2e-5, |error of GELU| <= 1.1e-6: an order of magnitude below the fp16 resolution of the output). With
// z = |x| / sqrt2 clamped to 4.3 (erfc(4.3) = 1.2e-9):  gelu(x) = max(x, 0) - 0.5 |x| erfc(z).
// The previous Abramowitz-Stegun 7.1.26 form needed rcp + ex2; at K = 320 the GEGLU epilogue (16 K outputs per tile and
// CTA) kept the 16-per-clock MUFU pipe busy for 2048 clocks against 2560 clocks of MMA.
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = fminf(fabsf(x) * 0.70710678118654752f, 4.3f);
  float q = fmaf(1.686094986e-05f, z, -4.376256625e-04f);
  q = fmaf(q, z, 4.960034474e-03f);
  q = fmaf(q, z, -3.321249048e-02f);
  q = fmaf(q, z, 1.515097036e-01f);
  q = fmaf(q, z, 9.176268788e-01f);
  q = fmaf(q, z, 1.627959694e+00f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-q * z));
  return fmaxf(x, 0.f) - z * 0.70710678118654752f * e;
}

template <int BN, int EPI, int CG, int NACC>
__global__ void __launch_bounds__(320, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
            const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmOut,
            const __grid_constant__ CUtensorMap tmRes, const GemmParams p) {
  using Cfg = GemmCfg<BN, CG, NACC>;
  constexpr int STAGES = Cfg::STAGES;
  griddep_launch_dependents();   // PDL: the next kernel may be scheduled; it waits for this one in ITS griddep_wait()
  // CG == 2: the CTAs of a pair (cluster of 2) work on two vertically adjacent 128-row tiles with ONE M=256 MMA issued
  // by the leader (rank 0). `cta_rank` selects this CTA's A rows and its half of the B tile.
  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * Cfg::A_BYTES;
  uint8_t* smem_epi = smem + STAGES * Cfg::STAGE_BYTES;   // 1024-aligned: per warp [2 KB out | 2 KB residual]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_epi + Cfg::EPI_STAGING);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;  // [3] one per accumulator slot (NACC == 1 uses two)
  uint64_t* res_bar = tmem_empty + 3;   // [8] one per epilogue warp
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(res_bar + 8);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work items: tiles (CG == 1) or pair-tiles of 2 x 128 rows (CG == 2); every CTA of a pair walks the same sequence
  const int n_groups = p.num_n_tiles / NACC;   // NACC adjacent BN-wide weight slabs form one work item
  const int num_tiles = (p.num_m_tiles / CG) * n_groups;
  const int first_tile = blockIdx.x / CG;
  const int tile_stride = gridDim.x / CG;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmB);
    if (p.kb_src2 > 0) tma_prefetch_desc(&tmA2);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) mbar_init(&tmem_full[s], 1);
    for (int s = 0; s < 3; ++s) mbar_init(&tmem_empty[s], 8 * CG);   // CG == 2: the leader collects both CTAs' warps
    for (int s = 0; s < 8; ++s) mbar_init(&res_bar[s], 1);
    if (p.tma_epi) {
      tma_prefetch_desc(&tmOut);
      if (p.residual != nullptr) tma_prefetch_desc(&tmRes);
    }
    fence_mbar_init();
  }
  if (CG == 2) cluster_sync();   // barrier inits visible cluster-wide before any remote arrive / 2-SM TMA
  if (warp == 1) {
    if (CG == 2) tmem_alloc_2sm<Cfg::TMEM_COLS>(tmem_ptr);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // everything above (barriers, TMEM, descriptor prefetch) is independent of the previous kernel's data; from here on the
  // TMA loads / epilogue reads touch it: wait until the previous kernel of the stream has completed (PDL)
  griddep_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (warp-uniform loop, elected lane
    // issues; tap / channel-block indices advance incrementally instead of by per-k-block integer division)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_stride) {
        const int m_tile = (tile / n_groups) * CG + (int)cta_rank;
        const int n_tile = (tile % n_groups) * NACC;
        int n0 = 0, y0 = 0, x0 = 0;
        if (p.a_mode != A_GEMM) {
          const int per_frame = p.tiles_x * p.tiles_y;
          const int tn = m_tile / per_frame;
          const int rem = m_tile % per_frame;
          n0 = tn * p.bn;
          y0 = (rem / p.tiles_x) * p.bh;
          x0 = (rem % p.tiles_x) * p.bw;
        }
        int within = 0, kx = 0, ky = 0;   // channel block inside the tap; tap = (ky, kx)
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            if (p.debug == 1) {   // timing experiment: no loads at all, the MMA consumes stale shared memory
              if (CG == 1 || cta_rank == 0) mbar_arrive(&full_bar[stage]);
            } else {
            // CG == 2: only the leader arms its barrier, with the bytes of BOTH CTAs (their TMA loads signal it)
            // debug 3 / 4 (timing experiments, garbage results): odd k-blocks skip the B / the A load, i.e. 19 % / 31 % less
            // L2 -> shared-memory traffic at an unchanged MMA schedule
            const bool load_a = !(p.debug == 4 && (kb & 1)), load_b = !(p.debug == 3 && (kb & 1));
            if (CG == 1 || cta_rank == 0)
              mbar_arrive_expect_tx(&full_bar[stage], CG * ((load_a ? Cfg::A_BYTES : 0) + (load_b ? Cfg::B_BYTES : 0)));
            void* a_dst = smem_a + stage * Cfg::A_BYTES;
            void* b_dst = smem_b + stage * Cfg::B_BYTES;
            const bool second = within >= p.kb_src1;
            const CUtensorMap* am = second ? &tmA2 : &tmA1;
            const int c0 = (second ? within - p.kb_src1 : within) * Cfg::BK;
            if (!load_a) {
            } else if (p.a_mode == A_GEMM) {
              if (CG == 2) tma_load_2d_2sm(am, &full_bar[stage], a_dst, c0, m_tile * Cfg::BM);
              else tma_load_2d(am, &full_bar[stage], a_dst, c0, m_tile * Cfg::BM);
            } else if (p.a_mode == A_CONV_S1) {
              if (CG == 2) tma_load_4d_2sm(am, &full_bar[stage], a_dst, c0, x0 + kx - 1, y0 + ky - 1, n0);
              else tma_load_4d(am, &full_bar[stage], a_dst, c0, x0 + kx - 1, y0 + ky - 1, n0);
            } else {
              // input pixel = 2*o + k - 1  ->  k=0: (o-1, phase 1), k=1: (o, phase 0), k=2: (o, phase 1)
              const int px = (kx == 1) ? 0 : 1, dx = (kx == 0) ? -1 : 0;
              const int py = (ky == 1) ? 0 : 1, dy = (ky == 0) ? -1 : 0;
              if (CG == 2) tma_load_5d_2sm(am, &full_bar[stage], a_dst, px * p.C1 + c0, x0 + dx, py, y0 + dy, n0);
              else tma_load_5d(am, &full_bar[stage], a_dst, px * p.C1 + c0, x0 + dx, py, y0 + dy, n0);
            }
            if (!load_b) {
            } else if (CG == 2) {
#pragma unroll
              for (int a = 0; a < NACC; ++a)
                tma_load_2d_2sm(&tmB, &full_bar[stage], static_cast<uint8_t*>(b_dst) + a * Cfg::B_SLAB, kb * Cfg::BK,
                                (n_tile + a) * BN + (int)cta_rank * (BN / 2));
            } else
              tma_load_2d(&tmB, &full_bar[stage], b_dst, kb * Cfg::BK, n_tile * BN);
            }
          }
          __syncwarp();
          if (++within == p.kb_src1 + p.kb_src2) {
            within = 0;
            if (++kx == 3) { kx = 0; ++ky; }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // The whole warp walks the loop with warp-uniform state (so ptxas keeps stage / descriptor math in uniform
    // registers instead of per-instruction R2UR broadcast loops); one elected lane issues tcgen05.mma / commit.
    if (cta_rank == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(128 * CG, BN);
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t a_base = smem_u32(smem_a), b_base = smem_u32(smem_b);
      uint32_t use0 = 0, use1 = 0, use2 = 0;   // completed uses of each accumulator slot (parity of its empty barrier)
      uint32_t it = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_stride, ++it) {
        // accumulator slots of this work item: NACC == 1 ping-pongs 0 / 1, NACC == 2 rotates through three
        const int s0 = NACC == 2 ? (int)((2 * it) % 3) : (int)(it & 1);
        const int s1 = NACC == 2 ? (int)((2 * it + 1) % 3) : s0;
        auto wait_slot = [&](int s) {
          uint32_t& u = s == 0 ? use0 : (s == 1 ? use1 : use2);
          mbar_wait(&tmem_empty[s], (u & 1) ^ 1);
          ++u;
        };
        wait_slot(s0);
        tc_fence_after();
        const uint32_t d0 = tmem_base + s0 * BN, d1 = tmem_base + s1 * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = umma_desc_k_sw128(a_base + stage * Cfg::A_BYTES);
          const uint64_t db = umma_desc_k_sw128(b_base + stage * Cfg::B_BYTES);
          if (elect_one()) {
            if (p.debug != 2)
#pragma unroll
            for (int k = 0; k < Cfg::BK / 16; ++k) {
              // advance 16 fp16 = 32 B along K inside the 128 B swizzle atom: +2 in the (>>4) start-address field
              if (CG == 2) umma_f16_ss_2sm(d0, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
              else umma_f16_ss(d0, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            }
          }
          if (NACC == 2) {
            if (kb == 0) {   // the second slot belonged to the previous item's first half: wait for its drain only now
              wait_slot(s1);
              tc_fence_after();
            }
            const uint64_t db1 = umma_desc_k_sw128(b_base + stage * Cfg::B_BYTES + Cfg::B_SLAB);
            if (elect_one()) {
              if (p.debug != 2)
#pragma unroll
              for (int k = 0; k < Cfg::BK / 16; ++k) umma_f16_ss_2sm(d1, da + 2 * k, db1 + 2 * k, idesc, (kb | k) != 0);
            }
          }
          if (elect_one()) {
            if (CG == 2) {
              umma_commit_2sm_mc(&empty_bar[stage], 3);                            // frees the stage in both CTAs
              if (kb == p.num_kb - 1) umma_commit_2sm_mc(&tmem_full[it & 1], 3);    // wakes both CTAs' epilogues
            } else {
              umma_commit(&empty_bar[stage]);
              if (kb == p.num_kb - 1) umma_commit(&tmem_full[it & 1]);
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..5)
    const int lane_group = warp & 3;  // TMEM lanes [32*lane_group, +32) are accessible to this warp
    const int col_half = (warp - 2) >> 2;  // the two warps of a lane quarter take alternating 32-column chunks
    const int row = lane_group * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    if (p.tma_epi) {
      // ---------------------------------------------------------------- TMA epilogue
      // Each warp owns rows [32*lane_group, +32) of the tile and every other 32-output-column chunk. A chunk travels
      // TMEM -> registers -> (bias / residual / GEGLU) -> fp16 -> this warp's 2 KB shared box (64B swizzle: bank-conflict
      // free row-per-thread writes) -> one TMA store; the residual chunk arrives the same way through a TMA load that
      // is issued one chunk ahead. No per-thread global memory instructions: row-per-thread LDG/STG touched 32
      // different cache lines per instruction and made the small-K GEMMs L1-wavefront bound.
      constexpr int ACC_PER_CHUNK = (EPI == EPI_GEGLU) ? 64 : 32;
      constexpr int NCHUNK = BN / ACC_PER_CHUNK;
      const int ew = warp - 2;
      uint8_t* obuf0 = smem_epi + ew * 4096;
      uint8_t* rbuf = obuf0 + 2048;
      // Without a residual the second 2 KB box of this warp is free: the output staging is then DOUBLE-buffered, so a chunk's
      // fp16 tile can be written while the TMA store of the previous chunk is still reading the other box (the K = 320
      // consumers are latency-bound in the epilogue — ncu: issue 28 % / 54 % active, tensor 45 % / 52 % — and every chunk used
      // to wait for the previous store to drain).
      uint32_t ochunk = 0;
      uint64_t* rbar = &res_bar[ew];
      uint32_t rphase = 0;
      const bool has_res = (EPI == EPI_LINEAR) && p.residual != nullptr;
      const int sw = (lane >> 1) & 3;                       // 64B-swizzle XOR term of this thread's row
      const int r0 = lane_group * 32;
      // LayerNorm-folding consumers: rstd of this thread's row in the NEXT tile
      float ln_next = 1.f;
      auto ln_prefetch = [&](int tile_) {
        if (tile_ >= num_tiles) return;
        const long long mm = (long long)((tile_ / n_groups) * CG + (int)cta_rank) * Cfg::BM + r0 + lane;   // A_GEMM rows
        ln_next = mm < p.M ? __ldg(p.ln_rstd + mm) : 1.f;
      };
      if (p.ln_rstd != nullptr) ln_prefetch(first_tile);
      uint32_t it = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_stride, ++it) {
        const int m_tile = (tile / n_groups) * CG + (int)cta_rank;
        const int n_tile = (tile % n_groups) * NACC;
        // accumulator slots of this work item (same rotation as the MMA issuer)
        const int s0 = NACC == 2 ? (int)((2 * it) % 3) : (int)(it & 1);
        const int s1 = NACC == 2 ? (int)((2 * it + 1) % 3) : s0;
        // coordinates of this warp's 32-row box
        int cy = 0, cx = 0, cn = 0;
        long long m = 0;
        bool row_ok = true;
        if (p.a_mode == A_GEMM) {
          cy = m_tile * Cfg::BM + r0;
          m = (long long)cy + lane;
          row_ok = m < p.M;
        } else {
          const int per_frame = p.tiles_x * p.tiles_y;
          const int tn = m_tile / per_frame;
          const int rem = m_tile % per_frame;
          cn = tn * p.bn + r0 / (p.bh * p.bw);
          cy = (rem / p.tiles_x) * p.bh + (r0 / p.bw) % p.bh;
          cx = (rem % p.tiles_x) * p.bw + r0 % p.bw;
          const int n = tn * p.bn + row / (p.bh * p.bw);
          const int y = (rem / p.tiles_x) * p.bh + (row / p.bw) % p.bh;
          const int x = (rem % p.tiles_x) * p.bw + row % p.bw;
          row_ok = (n < p.Nf) && (y < p.Ho) && (x < p.Wo);
          m = ((long long)n * p.Ho + y) * p.Wo + x;
        }
        const float* bias_row = nullptr;
        if (p.bias != nullptr) bias_row = p.bias + (row_ok ? (m / p.bias_group_rows) : 0) * p.bias_ld;
        // LayerNorm folding (consumer): the row's rstd, requested one tile ago (with K = 320 the epilogue is the critical
        // path: a load issued at the top of the tile is fully exposed)
        float ln_a = 1.f;
        if (p.ln_rstd != nullptr) {
          ln_a = ln_next;
          ln_prefetch(tile + tile_stride);
        }
        float rs_s = 0.f, rs_q = 0.f;   // producer: this warp's share of the row's {sum, sumsq}
        const bool want_stats = (EPI == EPI_LINEAR) && (p.row_stat_out != nullptr || p.col_stat_out != nullptr);
        auto load_res = [&](int chunk) {
          if (lane == 0) {
            mbar_arrive_expect_tx(rbar, 2048);
            const int col = n_tile * BN + chunk * 32;
            if (p.a_mode == A_GEMM) tma_load_2d(&tmRes, rbar, rbuf, col, cy);
            else tma_load_4d(&tmRes, rbar, rbuf, col, cx, cy, cn);
          }
        };
        if (has_res && col_half < NACC * NCHUNK) load_res(col_half);
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t t_lanes = tmem_base + (static_cast<uint32_t>(r0) << 16);
        bool released0 = false;
        auto release = [&](int slot) {   // this warp is done reading accumulator slot `slot`
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2) mbar_arrive_cluster(&tmem_empty[slot], 0);
            else mbar_arrive(&tmem_empty[slot]);
          }
        };
#pragma unroll 1
        for (int c = col_half; c < NACC * NCHUNK; c += 2) {
          if (NACC == 2 && c >= NCHUNK && !released0) {   // first slot drained: the next item's second half may start
            release(s0);
            released0 = true;
          }
          const uint32_t t_row = t_lanes + (c < NCHUNK ? s0 : s1) * BN - (c < NCHUNK ? 0 : NCHUNK) * ACC_PER_CHUNK;
          const int acol = n_tile * BN + c * ACC_PER_CHUNK;       // first accumulator (weight-row) column
          float v[32];
          if (EPI == EPI_GEGLU) {
            uint32_t r[64];
            tmem_ld_32x32b_x32(t_row + c * 64, r);
            tmem_ld_32x32b_x32(t_row + c * 64 + 32, r + 32);
            tmem_ld_wait();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              float bv[16], bg[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) { bv[j] = 0.f; bg[j] = 0.f; }
              if (bias_row != nullptr) {
                const float4* b4 = reinterpret_cast<const float4*>(bias_row + acol + h * 32);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const float4 a = __ldg(b4 + j), g = __ldg(b4 + 4 + j);
                  bv[4 * j] = a.x; bv[4 * j + 1] = a.y; bv[4 * j + 2] = a.z; bv[4 * j + 3] = a.w;
                  bg[4 * j] = g.x; bg[4 * j + 1] = g.y; bg[4 * j + 2] = g.z; bg[4 * j + 3] = g.w;
                }
              }
#pragma unroll
              for (int j = 0; j < 16; ++j)
                v[h * 16 + j] = fmaf(__uint_as_float(r[h * 32 + j]), ln_a, bv[j]) *
                                gelu_erf(fmaf(__uint_as_float(r[h * 32 + 16 + j]), ln_a, bg[j]));
            }
          } else {
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_row + c * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            if (p.ln_rstd != nullptr) {   // v = rstd * acc + bias (the folded beta.W^T + b: always present)
              const float4* b4 = reinterpret_cast<const float4*>(bias_row + acol);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 b = __ldg(b4 + j);
                v[4 * j + 0] = fmaf(v[4 * j + 0], ln_a, b.x);
                v[4 * j + 1] = fmaf(v[4 * j + 1], ln_a, b.y);
                v[4 * j + 2] = fmaf(v[4 * j + 2], ln_a, b.z);
                v[4 * j + 3] = fmaf(v[4 * j + 3], ln_a, b.w);
              }
            } else if (bias_row != nullptr) {
              const float4* b4 = reinterpret_cast<const float4*>(bias_row + acol);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 b = __ldg(b4 + j);
                v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
              }
            }
            if (EPI == EPI_GELU) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
            }
            if (has_res) {
              mbar_wait(rbar, rphase);
              rphase ^= 1;
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint4 u = *reinterpret_cast<const uint4*>(rbuf + lane * 64 + ((q ^ sw) << 4));
                const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const float2 f = __half22float2(h2[j]);
                  v[q * 8 + 2 * j] += f.x;
                  v[q * 8 + 2 * j + 1] += f.y;
                }
              }
            }
          }
          // the TMA store that last read the staging box we are about to overwrite must have finished reading it
          const bool dbl = !has_res && p.epi_double;
          uint8_t* obuf = (dbl && (ochunk & 1)) ? rbuf : obuf0;
          ++ochunk;
          if (lane == 0) {
            if (dbl) tma_store_wait_read<1>();
            else tma_store_wait_read<0>();
          }
          __syncwarp();
          if (want_stats && !row_ok) {   // rows past the end of the tensor are clipped by the store; keep them out of the sums
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            __half2 o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = __floats2half2_rn(v[q * 8 + 2 * j], v[q * 8 + 2 * j + 1]);
            if (EPI == EPI_LINEAR && p.row_stat_out != nullptr) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 f = __half22float2(o[j]);
                rs_s += f.x + f.y;
                rs_q = fmaf(f.x, f.x, fmaf(f.y, f.y, rs_q));
              }
            }
            *reinterpret_cast<uint4*>(obuf + lane * 64 + ((q ^ sw) << 4)) = *reinterpret_cast<uint4*>(o);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (EPI == EPI_LINEAR && p.col_stat_out != nullptr) {
            // column sums over the 32 rows of this warp's box, read back from the staged fp16 tile: lane = (row parity,
            // half2 column), 16 conflict-free 4-byte loads per lane, then the two row parities are added
            const int hc = lane & 15, rp = lane >> 4;
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
            for (int rr = 0; rr < 16; ++rr) {
              const int rw = 2 * rr + rp;
              const uint32_t u = *reinterpret_cast<const uint32_t*>(
                  obuf + rw * 64 + ((((hc >> 2) ^ ((rw >> 1) & 3))) << 4) + ((hc & 3) << 2));
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u));
              s0 += f.x; q0 = fmaf(f.x, f.x, q0);
              s1 += f.y; q1 = fmaf(f.y, f.y, q1);
            }
            s0 += __shfl_xor_sync(0xffffffffu, s0, 16);
            q0 += __shfl_xor_sync(0xffffffffu, q0, 16);
            s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
            q1 += __shfl_xor_sync(0xffffffffu, q1, 16);
            if (lane < 16) {
              float4* dst = reinterpret_cast<float4*>(p.col_stat_out + (long long)(m_tile * 4 + lane_group) * p.col_stat_ld +
                                                      n_tile * BN + c * 32 + 2 * hc);
              *dst = make_float4(s0, q0, s1, q1);
            }
          }
          if (has_res && c + 2 < NACC * NCHUNK) load_res(c + 2);      // rbuf fully consumed by every lane (syncwarp above)
          if (lane == 0) {
            const int ocol = n_tile * (BN / (EPI == EPI_GEGLU ? 2 : 1)) + c * 32;
            if (p.a_mode == A_GEMM) tma_store_2d(&tmOut, obuf, ocol, cy);
            else tma_store_4d(&tmOut, obuf, ocol, cx, cy, cn);
            tma_store_commit();
          }
        }
        if (NACC == 2 && !released0) release(s0);
        release(s1);
        if (EPI == EPI_LINEAR && p.row_stat_out != nullptr && row_ok)
          p.row_stat_out[(long long)(2 * (tile % n_groups) + col_half) * p.row_stat_ld + m] = make_float2(rs_s, rs_q);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (lane == 0) tma_store_wait_all<0>();   // stores must complete before the CTA (and its smem) goes away
    } else
    for (int tile = first_tile; tile < num_tiles; tile += tile_stride) {   // legacy direct-store epilogue (NACC == 1 only)
      const int m_tile = (tile / n_groups) * CG + (int)cta_rank;
      const int n_tile = tile % n_groups;
      // output row of this thread
      long long m;
      bool row_ok;
      if (p.a_mode == A_GEMM) {
        m = (long long)m_tile * Cfg::BM + row;
        row_ok = m < p.M;
      } else {
        const int per_frame = p.tiles_x * p.tiles_y;
        const int tn = m_tile / per_frame;
        const int rem = m_tile % per_frame;
        const int n = tn * p.bn + row / (p.bh * p.bw);
        const int y = (rem / p.tiles_x) * p.bh + (row / p.bw) % p.bh;
        const int x = (rem % p.tiles_x) * p.bw + row % p.bw;
        row_ok = (n < p.Nf) && (y < p.Ho) && (x < p.Wo);
        m = ((long long)n * p.Ho + y) * p.Wo + x;
      }
      const float* bias_row = nullptr;
      if (p.bias != nullptr) {
        const long long g = row_ok ? (m / p.bias_group_rows) : 0;
        bias_row = p.bias + g * p.bias_ld;
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + acc * BN + (static_cast<uint32_t>(lane_group * 32) << 16);
#pragma unroll 1
      for (int c = col_half; c < BN / 32; c += 2) {
        const int ncol = n_tile * BN + c * 32;  // column in weight-row space
        // issue the residual loads first so that their latency overlaps the TMEM load
        uint4 res4[4];
        const bool vec_ok = (ncol + 32 <= p.n_valid) && ((p.ldo & 7) == 0);
        const bool res_vec = EPI == EPI_LINEAR && p.residual != nullptr && row_ok && vec_ok && (p.ldr & 7) == 0;
        if (res_vec) {
          const uint4* r4 = reinterpret_cast<const uint4*>(p.residual + m * p.ldr + ncol);
#pragma unroll
          for (int q = 0; q < 4; ++q) res4[q] = __ldg(r4 + q);
        }
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_row + c * 32, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (bias_row != nullptr) {
          const float4* b4 = reinterpret_cast<const float4*>(bias_row + ncol);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = __ldg(b4 + j);
            v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
          }
        }
        if (EPI == EPI_GELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
        }
        if (EPI == EPI_GEGLU) {
          // interleaved weights: columns [0,16) = value half, [16,32) = gate half of the same 16 outputs
          const int ocol = ncol >> 1;
          if (row_ok) {
            __half2 o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float a0 = v[2 * j] * gelu_erf(v[16 + 2 * j]);
              const float a1 = v[2 * j + 1] * gelu_erf(v[16 + 2 * j + 1]);
              o[j] = __floats2half2_rn(a0, a1);
            }
            __half* dst = p.out + m * p.ldo + ocol;
            if (ocol + 16 <= p.n_valid && (p.ldo & 7) == 0) {
              uint4* d4 = reinterpret_cast<uint4*>(dst);
              d4[0] = *reinterpret_cast<uint4*>(&o[0]);
              d4[1] = *reinterpret_cast<uint4*>(&o[4]);
            } else {
              const __half* oh = reinterpret_cast<const __half*>(o);
              for (int j = 0; j < 16; ++j)
                if (ocol + j < p.n_valid) dst[j] = oh[j];
            }
          }
        } else {
          if (row_ok) {
            if (p.residual != nullptr) {
              if (res_vec) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const __half2* h2 = reinterpret_cast<const __half2*>(&res4[q]);
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 f = __half22float2(h2[j]);
                    v[q * 8 + 2 * j] += f.x;
                    v[q * 8 + 2 * j + 1] += f.y;
                  }
                }
              } else {
                const __half* rs = p.residual + m * p.ldr + ncol;
                for (int j = 0; j < 32; ++j)
                  if (ncol + j < p.n_valid) v[j] += __half2float(rs[j]);
              }
            }
            __half* dst = p.out + m * p.ldo + ncol;
            if (p.out_f32) {
              float* dstf = reinterpret_cast<float*>(p.out) + m * p.ldo + ncol;
              for (int j = 0; j < 32; ++j)
                if (ncol + j < p.n_valid) dstf[j] = v[j];
            } else if (vec_ok) {
              uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                __half2 o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) o[j] = __floats2half2_rn(v[q * 8 + 2 * j], v[q * 8 + 2 * j + 1]);
                d4[q] = *reinterpret_cast<uint4*>(o);
              }
            } else {
              for (int j = 0; j < 32; ++j)
                if (ncol + j < p.n_valid) dst[j] = __float2half_rn(v[j]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2) mbar_arrive_cluster(&tmem_empty[acc], 0);
        else mbar_arrive(&tmem_empty[acc]);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync();   // no CTA of the pair may exit (or free TMEM) while its peer can still signal it
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
template <int BN, int EPI, int CG, int NACC = 1>
static int launch_gemm(const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap& to,
                       const CUtensorMap& tr, const GemmParams& p, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, CG, NACC>;
  static bool attr_set = false;
  if (!attr_set) {
    AP_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel<BN, EPI, CG, NACC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int items = (p.num_m_tiles / CG) * (p.num_n_tiles / NACC);
  const int max_ctas = (num_sms() / CG) * CG;
  const int grid = items * CG < max_ctas ? items * CG : max_ctas;
  {
    cudaError_t le = launch_pdl(gemm_kernel<BN, EPI, CG, NACC>, dim3(grid), dim3(320), (size_t)Cfg::SMEM_BYTES, stream, CG, a1,
                                a2, b, to, tr, p);
    if (le != cudaSuccess) return fail(AP_ERR_CUDA, "gemm launch: %s", cudaGetErrorString(le));
  }
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

// Tile-width choice: wider tiles re-use the A operand more (less L2 traffic per FLOP) but give fewer tiles; small-M
// problems (16x16 / 8x8 levels) prefer narrower tiles to fill the 148 SMs and reduce wave-quantisation loss.
// geglu (also used for GELU): only tiles that are multiples of 64 columns
static int pick_bn(int N, int forced, long long m_tiles, bool geglu = false) {
  if (forced > 0) return forced;
  const int cand[5] = {256, 160, 128, 64, 32};
  const double quality[5] = {1.00, 0.95, 0.90, 0.70, 0.45};
  int best = -1;
  double best_score = -1.0;
  const int sms = num_sms();
  for (int i = 0; i < 5; ++i) {
    if (N % cand[i] != 0) continue;
    if (geglu && cand[i] % 64 != 0) continue;   // a GEGLU output chunk needs 64 accumulator columns
    const long long tiles = m_tiles * (N / cand[i]);
    const long long waves = (tiles + sms - 1) / sms;
    const double fill = (double)tiles / (double)(waves * sms);
    const double score = fill * quality[i];
    if (score > best_score + 1e-9) { best_score = score; best = cand[i]; }
  }
  return best;
}

// Wide (two-accumulator) tiles: used whenever the epilogue can use TMA and the work still fills the chip at least as well as
// with narrow tiles. The exposed part of the accumulator drain made K < 320 the only losing case on the UNet's shapes
// (whole-call replay 51.5 / 51.3 / 50.6 / 50.3 ms for a minimum of 30 / 20 / 10 / 5 k-blocks, same box).
static bool pick_wide(int bn, int epi, int cg, const GemmParams& p) {
  static const int env = getenv("AP_GEMM_WIDE") ? atoi(getenv("AP_GEMM_WIDE")) : -1;   // 0 = never, 1 = whenever legal
  if (env == 0) return false;
  if (!(bn == 160 && epi == EPI_LINEAR && cg == 2 && p.tma_epi && p.num_n_tiles % 2 == 0)) return false;
  if (env == 1) return true;
  static const int min_kb = getenv("AP_GEMM_WIDE_MINKB") ? atoi(getenv("AP_GEMM_WIDE_MINKB")) : 5;
  if (p.num_kb < min_kb) return false;
  const long long pairs = num_sms() / 2;
  const long long narrow = (long long)(p.num_m_tiles / 2) * p.num_n_tiles, wide = narrow / 2;
  const long long t_narrow = (narrow + pairs - 1) / pairs, t_wide = 2 * ((wide + pairs - 1) / pairs);
  // a wide work item takes ~0.8x the time of the two narrow ones it replaces: accept up to `slack` % more wave-units
  static const int slack = getenv("AP_GEMM_WIDE_SLACK") ? atoi(getenv("AP_GEMM_WIDE_SLACK")) : 25;
  return t_wide * 100 <= t_narrow * (100 + slack);
}

static int dispatch(int bn, int epi, int cg, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& b,
                    const CUtensorMap& to, const CUtensorMap& tr, const GemmParams& p, cudaStream_t stream) {
#define AP_CASE(BN_)                                                                     \
  case BN_:                                                                              \
    return epi == EPI_GEGLU ? launch_gemm<BN_, EPI_GEGLU, 1>(a1, a2, b, to, tr, p, stream) \
                            : launch_gemm<BN_, EPI_LINEAR, 1>(a1, a2, b, to, tr, p, stream);
#define AP_CASE2(BN_)                                                                    \
  case BN_:                                                                              \
    return epi == EPI_GEGLU ? launch_gemm<BN_, EPI_GEGLU, 2>(a1, a2, b, to, tr, p, stream) \
                            : launch_gemm<BN_, EPI_LINEAR, 2>(a1, a2, b, to, tr, p, stream);
  if (epi == EPI_GELU) {   // tiles that are multiples of 64 columns only (pick_bn never offers 160 / 32 for GELU)
    if (cg == 2) {
      if (bn == 256) return launch_gemm<256, EPI_GELU, 2>(a1, a2, b, to, tr, p, stream);
      if (bn == 128) return launch_gemm<128, EPI_GELU, 2>(a1, a2, b, to, tr, p, stream);
      return fail(AP_ERR_INVALID, "gemm: unsupported 2-CTA BLOCK_N %d with GELU", bn);
    }
    if (bn == 256) return launch_gemm<256, EPI_GELU, 1>(a1, a2, b, to, tr, p, stream);
    if (bn == 128) return launch_gemm<128, EPI_GELU, 1>(a1, a2, b, to, tr, p, stream);
    if (bn == 64) return launch_gemm<64, EPI_GELU, 1>(a1, a2, b, to, tr, p, stream);
    return fail(AP_ERR_INVALID, "gemm: unsupported BLOCK_N %d with GELU (multiples of 64 only)", bn);
  }
  if (cg == 2) {
    switch (bn) {
      AP_CASE2(256)
      case 160:
        if (pick_wide(bn, epi, cg, p)) return launch_gemm<160, EPI_LINEAR, 2, 2>(a1, a2, b, to, tr, p, stream);
        return launch_gemm<160, EPI_LINEAR, 2>(a1, a2, b, to, tr, p, stream);
      AP_CASE2(128)
      default:
        return fail(AP_ERR_INVALID, "gemm: unsupported 2-CTA BLOCK_N %d", bn);
    }
  }
  switch (bn) {
    AP_CASE(256)
    AP_CASE(160)
    AP_CASE(128)
    AP_CASE(64)
    AP_CASE(32)
    default:
      return fail(AP_ERR_INVALID, "gemm: unsupported BLOCK_N %d", bn);
  }
#undef AP_CASE
#undef AP_CASE2
}

// cta_group::2 is used when the work splits into pairs of 128-row tiles and the tile is wide enough to profit
static int pick_cg(int bn, int num_m_tiles, int num_n_tiles) {
  static const int env = getenv("AP_GEMM_CG") ? atoi(getenv("AP_GEMM_CG")) : 0;
  if (env == 1) return 1;
  if (num_m_tiles % 2 != 0) return 1;
  if (!(bn == 256 || bn == 160 || bn == 128)) return 1;
  if ((long long)num_m_tiles * num_n_tiles < 2LL * 74 && env != 2) return 1;   // too few pair-tiles to fill the chip
  return 2;
}

static int make_weight_map(CUtensorMap* tm, const void* w, int N, long long K, int bn_box) {
  const uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
  const uint64_t strides[1] = {(uint64_t)K * 2};
  const uint32_t box[2] = {64, (uint32_t)bn_box};
  return encode_tmap(tm, w, 2, dims, strides, box, true);
}

// Validates and copies the optional epilogue extensions into the kernel parameters (after tma_epi / tile counts are known).
static int apply_ext(GemmParams& p, const ap_epilogue_ext* ext, int epi, long long m_pad, int k_ln) {
  p.bias_ld = p.N;
  static const int epi_double = getenv("AP_GEMM_EPI_DOUBLE") ? atoi(getenv("AP_GEMM_EPI_DOUBLE")) : 1;
  p.epi_double = epi_double;
  if (ext == nullptr) return AP_OK;
  if (ext->bias_ld > 0) p.bias_ld = ext->bias_ld;
  const bool any = ext->row_stat_out || ext->col_stat_out || ext->ln_rstd;
  if (!any) return AP_OK;
  if (!p.tma_epi) return fail(AP_ERR_INVALID, "gemm: epilogue statistics / LayerNorm folding need the TMA epilogue (aligned fp16 out)");
  if (ext->row_stat_out) {
    if (epi != EPI_LINEAR) return fail(AP_ERR_INVALID, "gemm: row statistics are not available with GEGLU");
    if (ext->row_stat_ld < m_pad) return fail(AP_ERR_INVALID, "gemm: row_stat_ld %lld < padded M %lld", ext->row_stat_ld, m_pad);
    if (p.a_mode != A_GEMM) return fail(AP_ERR_INVALID, "gemm: row statistics only for plain GEMMs");
    p.row_stat_out = (float2*)ext->row_stat_out;
    p.row_stat_ld = ext->row_stat_ld;
  }
  if (ext->col_stat_out) {
    if (epi != EPI_LINEAR) return fail(AP_ERR_INVALID, "gemm: column statistics are not available with GEGLU");
    if (ext->col_stat_ld < p.N || (ext->col_stat_ld & 1)) return fail(AP_ERR_INVALID, "gemm: bad col_stat_ld %lld", ext->col_stat_ld);
    if ((reinterpret_cast<uintptr_t>(ext->col_stat_out) & 15) != 0) return fail(AP_ERR_INVALID, "gemm: col_stat_out must be 16-byte aligned");
    if (p.a_mode != A_GEMM && p.sub_n != 1)
      return fail(AP_ERR_INVALID, "conv3x3: column statistics need Ho*Wo %% 32 == 0 with 32-row sub-boxes inside one frame");
    p.col_stat_out = (float2*)ext->col_stat_out;
    p.col_stat_ld = ext->col_stat_ld;
  }
  if (ext->ln_rstd) {
    if (p.a_mode != A_GEMM) return fail(AP_ERR_INVALID, "gemm: LayerNorm folding only for plain GEMMs");
    if (p.bias == nullptr) return fail(AP_ERR_INVALID, "gemm: LayerNorm folding needs the folded bias (beta.W^T + b)");
    p.ln_rstd = ext->ln_rstd;
  }
  return AP_OK;
}

}  // namespace ap

using namespace ap;

extern "C" int ap_gemm_row_stat_parts(long long M, int N, int K, int flags, int block_n) {
  const int epi = (flags & AP_GEMM_GEGLU) ? EPI_GEGLU : ((flags & AP_GEMM_GELU) ? EPI_GELU : EPI_LINEAR);
  const int bn = pick_bn(N, block_n, (M + 127) / 128, epi != EPI_LINEAR);
  if (bn <= 0 || N % bn != 0) return fail(AP_ERR_INVALID, "gemm: N=%d not tileable (block_n=%d)", N, block_n);
  GemmParams p{};
  p.num_m_tiles = (int)((M + 127) / 128);
  p.num_n_tiles = N / bn;
  p.num_kb = (K + 63) / 64;
  p.tma_epi = 1;
  const int cg = pick_cg(bn, p.num_m_tiles, p.num_n_tiles);
  return p.num_n_tiles / (pick_wide(bn, epi, cg, p) ? 2 : 1);
}

extern "C" int ap_gemm_f16(const void* a, long long lda, int K1, const void* a2, long long lda2, int K2,
                           const void* w, long long M, int N, const float* bias, long long bias_group_rows,
                           const void* residual, long long ldr, void* out, long long ldo, int n_valid, int flags,
                           int block_n, void* stream, const ap_epilogue_ext* ext) {
  AP_REQUIRE(a && w && out, "gemm: null pointer");
  AP_REQUIRE(M > 0 && N > 0 && K1 > 0, "gemm: bad shape M=%lld N=%d K1=%d", M, N, K1);
  AP_REQUIRE(K1 % 64 == 0 || (a2 == nullptr), "gemm: K1 must be a multiple of 64 when a second source follows");
  AP_REQUIRE((lda % 8) == 0 && (a2 == nullptr || (lda2 % 8) == 0), "gemm: lda must be a multiple of 8 elements");
  AP_REQUIRE(!((flags & AP_GEMM_GEGLU) && (flags & AP_GEMM_GELU)), "gemm: AP_GEMM_GEGLU and AP_GEMM_GELU exclude each other");
  const int epi = (flags & AP_GEMM_GEGLU) ? EPI_GEGLU : ((flags & AP_GEMM_GELU) ? EPI_GELU : EPI_LINEAR);
  AP_REQUIRE(epi != EPI_GELU || residual == nullptr, "gemm: no residual with the GELU epilogue");
  const int bn = pick_bn(N, block_n, (M + 127) / 128, epi != EPI_LINEAR);
  AP_REQUIRE(epi == EPI_LINEAR || (bn > 0 && bn % 64 == 0), "gemm: GEGLU / GELU need a BLOCK_N multiple of 64");
  AP_REQUIRE(bn > 0 && N % bn == 0, "gemm: N=%d not tileable (block_n=%d)", N, block_n);
  const long long K = (long long)K1 + (a2 ? K2 : 0);
  AP_REQUIRE((K * 2) % 16 == 0, "gemm: K*2 bytes must be a multiple of 16");

  GemmParams p{};
  p.M = (int)M;
  p.N = N;
  p.num_m_tiles = (int)((M + 127) / 128);
  p.num_n_tiles = N / bn;
  p.a_mode = A_GEMM;
  p.kb_src1 = (K1 + 63) / 64;
  p.kb_src2 = a2 ? (K2 + 63) / 64 : 0;
  p.num_kb = p.kb_src1 + p.kb_src2;
  p.bias = bias;
  p.bias_group_rows = (int)(bias_group_rows > 0 ? (bias_group_rows > 0x7fffffff ? 0x7fffffff : bias_group_rows)
                                                : 0x7fffffff);
  p.residual = (const __half*)residual;
  p.ldr = (int)ldr;
  p.out = (__half*)out;
  p.ldo = (int)ldo;
  const int nout = epi == EPI_GEGLU ? N / 2 : N;
  p.n_valid = n_valid > 0 ? n_valid : nout;
  p.out_f32 = (flags & AP_GEMM_OUT_F32) ? 1 : 0;
  AP_REQUIRE(!(p.out_f32 && epi == EPI_GEGLU), "gemm: fp32 output is not available with GEGLU");

  CUtensorMap tmA1, tmA2, tmB;
  {
    const uint64_t dims[2] = {(uint64_t)K1, (uint64_t)M};
    const uint64_t strides[1] = {(uint64_t)lda * 2};
    const uint32_t box[2] = {64, 128};
    int rc = encode_tmap(&tmA1, a, 2, dims, strides, box, true);
    if (rc) return rc;
  }
  if (a2) {
    const uint64_t dims[2] = {(uint64_t)K2, (uint64_t)M};
    const uint64_t strides[1] = {(uint64_t)lda2 * 2};
    const uint32_t box[2] = {64, 128};
    int rc = encode_tmap(&tmA2, a2, 2, dims, strides, box, true);
    if (rc) return rc;
  } else {
    tmA2 = tmA1;
  }
  const int cg = pick_cg(bn, p.num_m_tiles, p.num_n_tiles);
  int rc = make_weight_map(&tmB, w, N, K, bn / cg);
  if (rc) return rc;
  // TMA epilogue whenever the output (and residual) satisfy TMA's 16-byte rules
  CUtensorMap tmOut = tmB, tmRes = tmB;
  const bool aligned_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ldo % 8) == 0 && (p.n_valid % 8) == 0;
  const bool aligned_res = residual == nullptr || ((reinterpret_cast<uintptr_t>(residual) & 15) == 0 && (ldr % 8) == 0);
  static const bool no_tma_epi = getenv("AP_GEMM_NO_TMA_EPI") != nullptr;
  if (!p.out_f32 && aligned_out && aligned_res && !no_tma_epi) {
    const uint64_t dims[2] = {(uint64_t)p.n_valid, (uint64_t)M};
    const uint32_t box[2] = {32, 32};
    const uint64_t so[1] = {(uint64_t)ldo * 2};
    if ((rc = encode_tmap(&tmOut, out, 2, dims, so, box, false, 2, 64))) return rc;
    if (residual) {
      const uint64_t sr[1] = {(uint64_t)ldr * 2};
      if ((rc = encode_tmap(&tmRes, residual, 2, dims, sr, box, false, 2, 64))) return rc;
    }
    p.tma_epi = 1;
  }
  if ((rc = apply_ext(p, ext, epi, (long long)p.num_m_tiles * 128, K1))) return rc;
  return dispatch(bn, epi, cg, tmA1, tmA2, tmB, tmOut, tmRes, p, (cudaStream_t)stream);
}

// 3x3 convolution, padding 1, stride 1 or 2, NHWC fp16, optional channel-concatenated second input.
extern "C" int ap_conv3x3_nhwc_f16(const void* x, int C1, const void* x2, int C2, int Nf, int H, int W, int stride,
                                   const void* w, int Cout, const float* bias, long long bias_group_rows,
                                   const void* residual, void* out, long long ldo, int n_valid, int block_n,
                                   void* stream, const ap_epilogue_ext* ext) {
  AP_REQUIRE(x && w && out, "conv3x3: null pointer");
  AP_REQUIRE(stride == 1 || stride == 2, "conv3x3: stride must be 1 or 2");
  AP_REQUIRE(C1 % 64 == 0 && (x2 == nullptr || C2 % 64 == 0), "conv3x3: channels must be multiples of 64 (pad)");
  AP_REQUIRE(stride == 1 || (H % 2 == 0 && W % 2 == 0), "conv3x3: stride 2 needs even H, W");
  const int Ho = H / stride, Wo = W / stride;
  const int bn_ = pick_bn(Cout, block_n, ((long long)Nf * Ho * Wo + 127) / 128);
  AP_REQUIRE(bn_ > 0 && Cout % bn_ == 0, "conv3x3: Cout=%d not tileable", Cout);

  // tile box: bw x bh x bn output pixels = 128 rows, bw | Wo, bh | Ho (powers of two)
  auto pow2_div = [](int v, int cap) { int d = 1; while (d * 2 <= cap && v % (d * 2) == 0) d *= 2; return d; };
  const int bw = pow2_div(Wo, 128);
  const int bh = pow2_div(Ho, 128 / bw);
  const int bnf = 128 / (bw * bh);

  GemmParams p{};
  p.Nf = Nf; p.Ho = Ho; p.Wo = Wo;
  p.bw = bw; p.bh = bh; p.bn = bnf;
  p.tiles_x = Wo / bw;
  p.tiles_y = Ho / bh;
  p.M = Nf * Ho * Wo;
  p.N = Cout;
  p.num_m_tiles = ((Nf + bnf - 1) / bnf) * p.tiles_x * p.tiles_y;
  p.num_n_tiles = Cout / bn_;
  p.a_mode = stride == 1 ? A_CONV_S1 : A_CONV_S2;
  p.kb_src1 = C1 / 64;
  p.kb_src2 = x2 ? C2 / 64 : 0;
  p.num_kb = 9 * (p.kb_src1 + p.kb_src2);
  p.C1 = C1;
  p.bias = bias;
  p.bias_group_rows = (int)(bias_group_rows > 0 ? (bias_group_rows > 0x7fffffff ? 0x7fffffff : bias_group_rows)
                                                : 0x7fffffff);
  p.residual = (const __half*)residual;
  p.ldr = (int)ldo;
  p.out = (__half*)out;
  p.ldo = (int)ldo;
  p.n_valid = n_valid > 0 ? n_valid : Cout;
  p.debug = getenv("AP_GEMM_DEBUG") ? atoi(getenv("AP_GEMM_DEBUG")) : 0;

  auto make_act_map = [&](CUtensorMap* tm, const void* base, int C) -> int {
    if (stride == 1) {
      const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)Nf};
      const uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
      const uint32_t box[4] = {64, (uint32_t)bw, (uint32_t)bh, (uint32_t)bnf};
      return encode_tmap(tm, base, 4, dims, strides, box, true);
    }
    // (phase_x * C + c, W/2, phase_y, H/2, Nf)
    const uint64_t dims[5] = {(uint64_t)2 * C, (uint64_t)W / 2, 2, (uint64_t)H / 2, (uint64_t)Nf};
    const uint64_t strides[4] = {(uint64_t)2 * C * 2, (uint64_t)W * C * 2, (uint64_t)2 * W * C * 2,
                                 (uint64_t)H * W * C * 2};
    const uint32_t box[5] = {64, (uint32_t)bw, 1, (uint32_t)bh, (uint32_t)bnf};
    return encode_tmap(tm, base, 5, dims, strides, box, true);
  };
  CUtensorMap tmA1, tmA2, tmB;
  int rc = make_act_map(&tmA1, x, C1);
  if (rc) return rc;
  if (x2) {
    rc = make_act_map(&tmA2, x2, C2);
    if (rc) return rc;
  } else {
    tmA2 = tmA1;
  }
  const int cg = pick_cg(bn_, p.num_m_tiles, p.num_n_tiles);
  rc = make_weight_map(&tmB, w, Cout, 9ll * (C1 + (x2 ? C2 : 0)), bn_ / cg);
  if (rc) return rc;
  CUtensorMap tmOut = tmB, tmRes = tmB;
  const bool aligned_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ldo % 8) == 0 && (p.n_valid % 8) == 0;
  const bool aligned_res = residual == nullptr || (reinterpret_cast<uintptr_t>(residual) & 15) == 0;
  static const bool no_tma_epi = getenv("AP_GEMM_NO_TMA_EPI") != nullptr;
  if (aligned_out && aligned_res && !no_tma_epi) {
    p.sub_w = bw < 32 ? bw : 32;
    p.sub_h = bh < 32 / p.sub_w ? bh : 32 / p.sub_w;
    p.sub_n = 32 / (p.sub_w * p.sub_h);
    const uint64_t dims[4] = {(uint64_t)p.n_valid, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)Nf};
    const uint64_t so[3] = {(uint64_t)ldo * 2, (uint64_t)Wo * ldo * 2, (uint64_t)Ho * Wo * ldo * 2};
    const uint32_t box[4] = {32, (uint32_t)p.sub_w, (uint32_t)p.sub_h, (uint32_t)p.sub_n};
    if ((rc = encode_tmap(&tmOut, out, 4, dims, so, box, false, 2, 64))) return rc;
    if (residual && (rc = encode_tmap(&tmRes, residual, 4, dims, so, box, false, 2, 64))) return rc;
    p.tma_epi = 1;
  }
  if ((rc = apply_ext(p, ext, EPI_LINEAR, (long long)p.num_m_tiles * 128, 0))) return rc;
  // entry e of the partials must belong to frame e / (Ho*Wo/32): tiles inside one frame, or whole frames per tile
  if (p.col_stat_out)
    AP_REQUIRE((Ho * Wo) % 32 == 0 && (p.bn == 1 || p.tiles_x * p.tiles_y == 1),
               "conv3x3: column statistics need Ho*Wo %% 32 == 0 and frame-major 32-row sub-boxes (Ho=%d Wo=%d)", Ho, Wo);
  return dispatch(bn_, EPI_LINEAR, cg, tmA1, tmA2, tmB, tmOut, tmRes, p, (cudaStream_t)stream);
}
