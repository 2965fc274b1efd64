// The ensemble MLP of a step as independent chains whose activations and gradients stay RESIDENT in shared memory.
//
// k_mlp_chain (gemm_chain.cuh) gives a CTA whole (row tile, member) chains, but every layer still hands its output to
// the next through global memory: the epilogue stores the tiled operand and the next layer copies it back in by TMA.
// Here a CTA runs one chain at a time through all of its phases,
//     fwd1 -> fwd2 -> fwd3 + head -> bwd3 -> bwd2 -> bwd1 (-> dE/dAEV, one unit per live column tile),
// and the A operand of every layer after the first is a 128-row image in shared memory (`res`, up to 8 K-blocks of
// [p1 | p2], SWIZZLE_64B -- the layout the UMMA descriptors read) that the previous layer's epilogue writes from
// registers.  Each K-block of that image has an mbarrier: the four warps that complete it arrive (after a proxy
// fence), and the MMA warp issues the next layer's K-block j as soon as barrier j has completed -- into the other
// TMEM accumulator, so the next layer's main loop runs under the current layer's epilogue.  Overwriting the image in
// place is safe: a layer's epilogue starts once its accumulator is full, i.e. after every MMA that read the image.
//
// What still touches global memory: the AEV operand (layer-1 forward, through the ring), the weights, act1 / act2
// (the forward epilogues of layers 1 and 2 also store them: the backward epilogues need CELU' -- the very thread that
// stored an element reads it back, so program order is all the ordering there is), e_member, and dE/dAEV (vector
// REDs, or per-member slabs).  The gradients g3, g2, g1 never leave the SM.
//
// Shared memory: [res | B-only ring] for phases 1-5, and for the layer-1 forward a ring of A + B stages over ALL of it
// (res is free until the fwd1 epilogue); every phase sizes its stages by its widest tile.  The producer drains the
// ring when the phase changes; both roles restart at slot 0 (parities per barrier in bit masks, as in k_mlp_fused).
// The host computes the plan (mlp.cu, resident_plan) and launches this kernel only where it fits: 2 x fp16 operands
// with hidden widths <= 256.
//
// Requirements (checked by the launcher): those of k_mlp_chain, one member per layer-1 backward unit.
#pragma once
#include "gemm_chain.cuh"

namespace ani {
namespace tc {

constexpr int RES_MAX_KB = TN_MAX / TK;                                   // 8 K-blocks of 32 columns
constexpr int RES_B_STAGE_BYTES = PARTS * TN_MAX * ROW_BYTES;            // phases 1-5: B only
constexpr int RES_AVAIL = FUSED_SMEM_BYTES - 1024;

struct ResidentArgs {
  int n_phases;            // 3 (forward only) or 6
  int res_kb;              // K-blocks of the resident image (widest hidden layer / 32)
  int epi[MAX_PHASES];
  Args ph[MAX_PHASES];
};

// one potentially blocking probe (the thread may be suspended for a while instead of spinning on issue slots the
// epilogue warps need)
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// bounded wait: false (and ANI_STATUS_INTERNAL raised, every later wait of the CTA given up at once) on a timeout
__device__ __forceinline__ bool mbar_wait_bounded(uint64_t* bar, uint32_t parity, int32_t* status, volatile int* abort) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  while (true) {
    if (mbar_try_wait(bar, parity)) return true;
    if (*abort) return false;
    if (clock64() - t0 > FUSED_SPIN_LIMIT) {
      if (status) atomicOr(status, ANI_STATUS_INTERNAL);
      *abort = 1;
      return false;
    }
  }
}

__global__ void __launch_bounds__(CHAIN_THREADS, 1) k_mlp_resident(const __grid_constant__ ResidentArgs F) {
  constexpr int NW = NUM_EPI_WARPS, C_MMA_WARP = NW, C_PROD_WARP = NW + 1;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ TileMap tms[MAX_PHASES];
  __shared__ int s_total_rt, s_units_per_chain;
  __shared__ volatile int s_abort;
  __shared__ float e_part[NW * 32];
  __shared__ __align__(16) float s_bias[2][TN_MAX];
  __shared__ __align__(16) float s_w4[2][TN_MAX];
  __shared__ __align__(8) uint64_t bars[2 * MAX_STAGES + 5 + RES_MAX_KB];
  uint64_t* full = bars;
  uint64_t* empty = bars + MAX_STAGES;
  uint64_t* tfull = bars + 2 * MAX_STAGES;
  uint64_t* tempty = bars + 2 * MAX_STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 4);
  uint64_t* rbar = bars + 2 * MAX_STAGES + 5;   // [K-block]: the resident image's K-block is complete (4 warps)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NP = F.n_phases;
  int32_t* status = F.ph[0].status;
  unsigned char* res = smem;
  unsigned char* small_ring = smem + F.res_kb * A_BLOCK_BYTES;

  if (lane == 0 && warp < NP) build_tile_map(F.ph[warp], tms[warp]);
  __syncthreads();
  if (threadIdx.x == 0) {
    s_abort = 0;
    s_total_rt = F.ph[0].layout_info[4 + F.ph[0].num_species];
    int last_ntn = 1;
    for (int s = 0; s < F.ph[0].num_species; ++s)
      if (tms[NP - 1].cnt_rt[s] > 0) last_ntn = max(last_ntn, tms[NP - 1].ntn[s]);
    s_units_per_chain = NP - 1 + last_ntn;
    // ring geometry per phase, from its widest tile: the layer-1 forward's A + B stages over all of the shared memory,
    // the other phases' B stages behind the resident image (a 160-column layer gets four stages where 256 gets two)
    for (int p = 0; p < NP; ++p) {
      int bmax = 32;
      for (int s = 0; s < F.ph[p].num_species; ++s)
        if (tms[p].cnt_rt[s] > 0) bmax = max(bmax, min(tms[p].tn[s], tms[p].n_eff[s]));
      tms[p].stage_bytes = PARTS * bmax * ROW_BYTES + (p == 0 ? A_BLOCK_BYTES : 0);
      const int region = p == 0 ? RES_AVAIL : RES_AVAIL - F.res_kb * A_BLOCK_BYTES;
      tms[p].stages = max(1, min(MAX_STAGES, region / tms[p].stage_bytes));
    }
    for (int i = 0; i < MAX_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], NW);
    }
    for (int i = 0; i < RES_MAX_KB; ++i) mbar_init(&rbar[i], 4);
    fence_barrier_init();
  }
  if (warp == C_MMA_WARP) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int M = F.ph[0].members;
  const int num_chains = s_total_rt * M, U = s_units_per_chain;
  // Chains in list order, CTA c taking c, c + G, ...: the row tiles are grouped by species in the model's species
  // order, whose networks (ANI-1x, ANI-2x) are widest first, so every CTA meets the long chains first and ends on
  // short ones.
  auto decode = [&](const ChainUnit& cu, int& p, Tile& tl) {
    p = min(cu.u, NP - 1);
    const int nt = cu.u - p;
    const int rt = cu.chain / M;
    const TileMap& tm = tms[p];
    int s = 0;
    while (s + 1 < F.ph[p].num_species && rt >= tm.first_rt[s] + tm.cnt_rt[s]) ++s;
    tl.s = s;
    tl.rt = rt;
    tl.mem = cu.chain - rt * M;
    tl.rt_last = tm.first_rt[s] + tm.cnt_rt[s] - 1;
    tl.n0 = nt * tm.tn[s];
    tl.bn = min(tm.tn[s], tm.n_eff[s] - tl.n0);
    return nt < tm.ntn[s] && rt >= tm.first_rt[s];
  };

  if (warp == C_PROD_WARP) {
    // ================================ producer (TMA) ================================
    uint32_t stage = 0, empty_par = 0xffffffffu;
    int geom = -1, STAGES = 1, STAGE_BYTES = 0;   // geometry = phase
    ChainWalk w;
    w.init(gridDim.x, blockIdx.x, 1, U, num_chains);
    ChainUnit cu;
    while (w.next(cu)) {
      int p;
      Tile tl;
      if (!decode(cu, p, tl)) continue;
      if (p != geom) {
        // every slot of the old geometry consumed: its MMAs (and, leaving phase 5, every MMA that read the resident
        // image) have completed before the new one's copies land on top of them.  (Costs nothing in the steady
        // state: the last MMAs of a phase complete before its epilogue starts, and the epilogue is where the next
        // phase's first copies are issued.)
        for (int s = 0; s < STAGES && geom >= 0; ++s) mbar_wait_bounded(&empty[s], (empty_par >> s) & 1u, status, &s_abort);
        geom = p;
        STAGES = tms[p].stages;
        STAGE_BYTES = tms[p].stage_bytes;
        stage = 0;
      }
      const Args& args = F.ph[p];
      const TileMap& tm = tms[p];
      const Species& sp = args.sp[tl.s];
      const int nkb = tm.kb_count >= 0 ? tm.kb_count : (sp.K + TK - 1) / TK;
      const int nkb_all = sp.b_kb_moff ? sp.b_kblocks : (sp.K + TK - 1) / TK;
      const int kb_boff = tl.mem * sp.b_kb_moff;
      const unsigned char* At = args.A + (size_t)tl.rt * args.a_kblocks * A_BLOCK_BYTES;   // layer 1: shared AEV tile
      const unsigned char* Bm =
          sp.Bt + (sp.b_kb_moff ? (size_t)0 : (size_t)tl.mem * sp.N * nkb_all * (PARTS * ROW_BYTES));
      const uint32_t b_bytes = (uint32_t)tl.bn * ROW_BYTES;
      const uint32_t a_bytes = p == 0 ? (uint32_t)A_BLOCK_BYTES : 0u;
      const bool dense = tm.nb_count < 0 || args.b_compact;
      const int n0p = tl.n0 / TN_MAX * TN_MAX, bnp = min(TN_MAX, (args.b_compact ? tm.n_eff[tl.s] : sp.N) - n0p);
      const int gq = lane / PARTS, gpart = lane % PARTS;
      size_t g_src = 0;
      int g_bns = 0;
      const bool g_active = !dense && lane < PARTS * (tl.bn / 32);
      if (g_active) {
        const int row0 = tm.nb[tl.n0 / 32 + gq] * 32;
        const int n0s = row0 / TN_MAX * TN_MAX;
        g_bns = min(TN_MAX, sp.N - n0s);
        g_src = (size_t)n0s * nkb_all * (PARTS * ROW_BYTES) + (size_t)(row0 - n0s) * ROW_BYTES +
                (size_t)gpart * g_bns * ROW_BYTES;
      }
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait_bounded(&empty[stage], (empty_par >> stage) & 1u, status, &s_abort);
        empty_par ^= 1u << stage;
        unsigned char* st = (p == 0 ? smem : small_ring) + stage * STAGE_BYTES;
        unsigned char* sb = st + a_bytes;
        const int kbi = tm.kb_count >= 0 ? tm.kb[kb] : kb;
        const int kbb = kbi + kb_boff;
        if (lane == 0) {
          mbar_arrive_expect_tx(&full[stage], a_bytes + PARTS * b_bytes);
          if (p == 0) bulk_g2s(st, At + (size_t)kbi * A_BLOCK_BYTES, A_BLOCK_BYTES, &full[stage]);
          if (dense) {
            if (tl.bn == bnp) {
              const unsigned char* bsrc = Bm + ((size_t)tl.n0 * nkb_all + (size_t)kbb * tl.bn) * (PARTS * ROW_BYTES);
              bulk_g2s(sb, bsrc, PARTS * b_bytes, &full[stage]);
            } else {
#pragma unroll
              for (int pc = 0; pc < PARTS; ++pc)
                bulk_g2s(sb + pc * b_bytes,
                         Bm + ((size_t)n0p * nkb_all + (size_t)kbb * bnp) * (PARTS * ROW_BYTES) +
                             (size_t)pc * bnp * ROW_BYTES + (size_t)(tl.n0 - n0p) * ROW_BYTES,
                         b_bytes, &full[stage]);
            }
          }
        }
        __syncwarp();
        if (g_active)
          bulk_g2s(sb + gpart * b_bytes + gq * 32 * ROW_BYTES, Bm + g_src + (size_t)kbb * g_bns * (PARTS * ROW_BYTES),
                   32 * ROW_BYTES, &full[stage]);
        __syncwarp();
        if (++stage == (uint32_t)STAGES) stage = 0;
      }
    }
  } else if (warp == C_MMA_WARP) {
    // ================================ MMA issuer ================================
    uint32_t stage = 0, full_par = 0u, acc = 0, acc_phase = 0, res_par = 0u;
    int geom = -1, STAGES = 1, STAGE_BYTES = 0;
    ChainWalk w;
    w.init(gridDim.x, blockIdx.x, 1, U, num_chains);
    ChainUnit cu;
    while (w.next(cu)) {
      int p;
      Tile tl;
      if (!decode(cu, p, tl)) continue;
      if (p != geom) {
        geom = p;
        STAGES = tms[p].stages;
        STAGE_BYTES = tms[p].stage_bytes;
        stage = 0;
      }
      const Args& args = F.ph[p];
      const TileMap& tm = tms[p];
      const int nkb = tm.kb_count >= 0 ? tm.kb_count : (args.sp[tl.s].K + TK - 1) / TK;
      const uint32_t idesc = make_idesc(tl.bn, TM);
      const uint32_t b_bytes = (uint32_t)tl.bn * ROW_BYTES;
      // the first unit of phases 1-5 reads the image the previous phase's epilogue is writing: K-block by K-block
      const bool wait_res = p > 0 && tl.n0 == 0;
      mbar_wait_bounded(&tempty[acc], acc_phase ^ 1, status, &s_abort);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * TN_MAX;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait_bounded(&full[stage], (full_par >> stage) & 1u, status, &s_abort);
        full_par ^= 1u << stage;
        if (wait_res) {
          mbar_wait_bounded(&rbar[kb], (res_par >> kb) & 1u, status, &s_abort);
          res_par ^= 1u << kb;
        }
        tc_fence_after();
        if (lane == 0) {
          uint32_t sa, sb;
          if (p == 0) {
            sa = smem_u32(smem + stage * STAGE_BYTES);
            sb = sa + A_BLOCK_BYTES;
          } else {
            sa = smem_u32(res + kb * A_BLOCK_BYTES);
            sb = smem_u32(small_ring + stage * STAGE_BYTES);
          }
          const uint64_t a1 = make_desc(sa), a2 = make_desc(sa + A_PART_BYTES);
          const uint64_t b1 = make_desc(sb), b2 = make_desc(sb + b_bytes);
#if !ANI_OPND_FP16X2
          const uint64_t a3 = make_desc(sa + 2 * A_PART_BYTES), b3 = make_desc(sb + 2 * b_bytes);
#endif
#pragma unroll
          for (int k = 0; k < TK / 16; ++k) {
            const uint64_t adv = (uint64_t)(k * 2);
#if ANI_OPND_FP16X2
            umma_f16(d_tmem, a2 + adv, b1 + adv, idesc, (kb | k) != 0);
            umma_f16(d_tmem, a1 + adv, b2 + adv, idesc, 1);
            umma_f16(d_tmem, a1 + adv, b1 + adv, idesc, 1);
#else
            umma_f16(d_tmem, a3 + adv, b1 + adv, idesc, (kb | k) != 0);
            umma_f16(d_tmem, a1 + adv, b3 + adv, idesc, 1);
            umma_f16(d_tmem, a2 + adv, b2 + adv, idesc, 1);
            umma_f16(d_tmem, a2 + adv, b1 + adv, idesc, 1);
            umma_f16(d_tmem, a1 + adv, b2 + adv, idesc, 1);
            umma_f16(d_tmem, a1 + adv, b1 + adv, idesc, 1);
#endif
          }
          umma_commit(&empty[stage]);
          if (kb == nkb - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++stage == (uint32_t)STAGES) stage = 0;
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else {
    // ================================ epilogue ================================
    uint32_t acc = 0, acc_phase = 0, buf = 0;
    float omax = 0.f;
    const int quad = warp & 3;
    ChainWalk w;
    w.init(gridDim.x, blockIdx.x, 1, U, num_chains);
    ChainUnit cu;
    while (w.next(cu)) {
      int p;
      Tile tl;
      if (!decode(cu, p, tl)) continue;
      const Args& args = F.ph[p];
      const TileMap& tm = tms[p];
      const int epi = F.epi[p];
      const Species& sp = args.sp[tl.s];
      if (epi == EPI_BIAS_CELU || epi == EPI_HEAD) {
        const int c = threadIdx.x;
        if (c < tl.bn) {
          // (the register-direct epilogue folds the output scale into the staged bias)
          s_bias[acc][c] = sp.bias[(size_t)tl.mem * sp.bias_mstride + tl.n0 + c] * (epi == EPI_BIAS_CELU ? args.out_scale : 1.0f);
          if (epi == EPI_HEAD) s_w4[acc][c] = sp.w4[(size_t)tl.mem * sp.N + c];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
      }
      // (every epilogue warp sees the same barrier phase: all of them run the tile or, after a timeout, none)
      if (mbar_wait_bounded(&tfull[acc], acc_phase, status, &s_abort)) {
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * TN_MAX;
        // act1 / act2 (phases 0, 1) are also stored for the backward epilogues; the gradients only live in `res`
        const bool c_store = p <= 1;
        int groups = 0;
        switch (epi) {
          case EPI_BIAS_CELU:
            tile_epilogue_direct<EPI_BIAS_CELU>(args, tl, tl.rt, sp, taddr, s_bias[acc], s_w4[acc], e_part, warp, lane,
                                                &tfull[acc], acc_phase, omax, true, res, rbar, c_store);
            break;
          case EPI_MUL_DCELU:
            tile_epilogue_direct<EPI_MUL_DCELU>(args, tl, tl.rt, sp, taddr, s_bias[acc], s_w4[acc], e_part, warp, lane,
                                                &tfull[acc], acc_phase, omax, true, res, rbar, c_store);
            break;
          case EPI_HEAD:
            tile_epilogue_direct<EPI_HEAD>(args, tl, tl.rt, sp, taddr, s_bias[acc], s_w4[acc], e_part, warp, lane,
                                           &tfull[acc], acc_phase, omax, true, res, rbar, c_store);
            break;
          default:
            tile_epilogue8<EPI_PLAIN>(args, tm, tl, sp, taddr, nullptr, 0, buf, s_bias[acc], s_w4[acc], e_part, warp, lane,
                                      &tfull[acc], acc_phase, omax, groups);
            break;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (ANI_OPND_FP16X2 && status && !(omax <= OPND_HALF_MAX)) atomicOr(status, ANI_STATUS_OPERAND_RANGE);
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == C_MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc
}  // namespace ani
