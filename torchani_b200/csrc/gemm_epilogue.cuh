// Register-direct epilogue of the tcgen05 GEMMs (gemm_tc.cuh / gemm_fused.cuh).
//
// Measured with the debug switches of k_gemm_tc (tools/mlp_probe.py, 9 999-atom water box, six launches 222 us):
// epilogue alone 165 us = launch floor ~48 + math 52 + split / shared-memory staging / proxy fence / TMA store 43
// + stored-activation loads 21, against ~79 us each for the copies alone and the MMAs alone -- the epilogue was the
// longest of the three pipelines.  This version
//   * writes the tiled operand straight from registers: a thread (= accumulator row) owns, per 16-column half and
//     piece, one aligned 32-byte sector of the SWIZZLE_64B image (its two 16-byte chunks are neighbours; rows with
//     (row >> 1) & 1 hold them in swapped order) -> one 256-bit store per half and piece, full sectors, no shared-memory
//     staging, no proxy fence, no bulk-store bookkeeping; the 64 KB of staging buffers go to the operand ring;
//   * reads the stored activation (EPI_MUL_DCELU) the same way, one 256-bit L2 load per half and piece;
//   * does the arithmetic on packed fp32 pairs (fma / mul / add .f32x2) with the power-of-two operand scales folded
//     into the constants -- bit-identical results (scaling by a power of two commutes with rounding).
// Completion for the data-flow launch: the stores are plain generic-proxy stores; the warp arrives in shared memory
// right after issuing them and the signal warp's gpu-scope fence + release-add publishes them (cumulativity through
// the cta-scope synchronisation, the pattern of a grid barrier).
#pragma once
#include "gemm_tc.cuh"

namespace ani {
namespace tc {

typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}
// one aligned 32-byte sector: two 16-byte chunks, q0 at the lower address
__device__ __forceinline__ void stg256(void* p, const uint4& q0, const uint4& q1) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(q0.x), "r"(q0.y), "r"(q0.z),
               "r"(q0.w), "r"(q1.x), "r"(q1.y), "r"(q1.z), "r"(q1.w)
               : "memory");
}
// (L2 only: the lines were written by another SM earlier in this launch, or by this one; never through this L1)
__device__ __forceinline__ void ldg256_cg(const void* p, uint4& q0, uint4& q1) {
  asm volatile("ld.global.cg.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(q0.x), "=r"(q0.y), "=r"(q0.z), "=r"(q0.w), "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w)
               : "l"(p)
               : "memory");
}
// sum of the PARTS 16-bit pieces of a column pair (smallest piece first) as a packed fp32 pair, still scaled
__device__ __forceinline__ f32x2 join_pair(const uint32_t (&w)[PARTS]) {
#if ANI_OPND_FP16X2
  const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&w[1]));
  const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&w[0]));
  return add2(pack2(lo.x, lo.y), pack2(hi.x, hi.y));
#else
  f32x2 acc = pack2(__uint_as_float(w[PARTS - 1] << 16), __uint_as_float(w[PARTS - 1] & 0xffff0000u));
#pragma unroll
  for (int p = PARTS - 2; p >= 0; --p) acc = add2(acc, pack2(__uint_as_float(w[p] << 16), __uint_as_float(w[p] & 0xffff0000u)));
  return acc;
#endif
}
// 8 consecutive accumulator columns of this thread's TMEM lane (asynchronous issue; tmem_ld_wait8 before use)
__device__ __forceinline__ void tmem_ld8_issue(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait8(uint32_t (&r)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])
               :
               : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& q) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
}
__device__ __forceinline__ uint32_t u4_word(const uint4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

// The epilogue of one tile, eight epilogue warps (thread = accumulator row; warps w and w + 4 share a TMEM lane quadrant
// and take alternate 32-column groups).  EPI_BIAS_CELU / EPI_MUL_DCELU / EPI_HEAD only (tiled outputs).
//   bias   shared memory, this tile's columns: bias * out_scale (EPI_BIAS_CELU) or plain (EPI_HEAD)
//   w4     shared memory, final-layer weights of this tile's columns (EPI_HEAD)
//   y_early  the stored activation may be read before the accumulator barrier (chained launches: it is older than
//            the launch; the data-flow launch orders it through that barrier)
//   res      (gemm_resident.cuh) the tiled output is also written to this shared-memory image of the 128-row tile,
//            K-block n0 / 32 + g at res + (n0 / 32 + g) * A_BLOCK_BYTES, and the four warps that complete K-block j
//            each arrive once on res_bar[j] (after a proxy fence: the next layer's MMAs read it)
//   c_store  false: no global stores of the tiled output (it only lives in `res`)
template <int EPI>
__device__ __forceinline__ void tile_epilogue_direct(const Args& args, const Tile& tl, int rt_mine, const Species& sp,
                                                     uint32_t taddr, const float* __restrict__ bias,
                                                     const float* __restrict__ w4, float* e_part, int warp, int lane,
                                                     uint64_t* tfull_bar, uint32_t tfull_parity, float& omax, bool y_early,
                                                     unsigned char* res, uint64_t* res_bar, bool c_store) {
  static_assert(EPI == EPI_BIAS_CELU || EPI == EPI_MUL_DCELU || EPI == EPI_HEAD, "tiled-output epilogues only");
  const int quad = warp & 3, half = warp >> 2;
  const int r_tile = quad * 32 + lane;
  // this row's two 32-byte sectors inside a 32-column block of one piece: half hh lives in sector hh ^ (sw >> 1), its
  // two chunks swapped when sw & 1 (SWIZZLE_64B: chunk position = chunk ^ ((row >> 1) & 3))
  const uint32_t sw = (uint32_t)(lane >> 1) & 3u;
  const bool swapped = sw & 1u;
  const uint32_t row_base = (uint32_t)(r_tile >> 3) * 512u + (uint32_t)(r_tile & 7) * 64u;
  const bool tiled_out = EPI != EPI_HEAD || args.want_backward;
  const bool g_out = tiled_out && c_store, s_out = tiled_out && res != nullptr;
  const uint32_t s_row = res ? smem_u32(res) + (uint32_t)(tl.n0 / TK) * A_BLOCK_BYTES + row_base : 0u;
  const int my_row = rt_mine * TM + r_tile;
  unsigned char* ct = reinterpret_cast<unsigned char*>(args.C) +
                      ((size_t)rt_mine * args.c_kblocks + (size_t)(tl.mem * sp.c_moff + tl.n0) / TK) * A_BLOCK_BYTES + row_base;
  const int ngroups = tl.bn / 32;
  const float os = args.out_scale;
  // constants with the operand scales folded in (all scales are powers of two)
  const float a_s = sp.acc_scale * (EPI == EPI_HEAD ? 1.0f : os);
  const f32x2 a2 = pack2(a_s, a_s);
  const float inv_alpha = 1.0f / args.alpha;
  const float kx = (EPI == EPI_HEAD ? 1.0f : 1.0f / os) * 1.4426950408889634f * inv_alpha;
  const float al = args.alpha * (EPI == EPI_HEAD ? 1.0f : os);
  const f32x2 kx2 = pack2(kx, kx), al2 = pack2(al, al), nal2 = pack2(-al, -al);
  const float cy = inv_alpha * args.y_inv_scale * a_s;   // EPI_MUL_DCELU: d = y > 0 ? a_s : fma(y, cy, a_s)
  const f32x2 cy2 = pack2(cy, cy);
  const f32x2 ia2 = pack2(inv_alpha, inv_alpha), one2 = pack2(1.0f, 1.0f);
  float seed = 0.f;
  bool row_valid = false;
  if (EPI == EPI_HEAD) {
    row_valid = args.row_atom[my_row] >= 0;
    seed = row_valid ? args.member_scale[tl.mem] * os : 0.f;
  }
  const f32x2 seed2 = pack2(seed, seed);
  f32x2 e_acc2 = pack2(0.f, 0.f);

  // stored activation of this row: per half one register set [piece][chunk], refilled for the same half of the warp's
  // next group as soon as it has been consumed (a whole group of epilogue math ahead)
  uint4 yq[2][PARTS][2];
  auto load_y = [&](int g, int hh, uint4 (&q)[PARTS][2]) {
    const unsigned char* src = ct + (size_t)g * A_BLOCK_BYTES + ((uint32_t)(hh ^ (int)(sw >> 1)) << 5);
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
      if (swapped)
        ldg256_cg(src + p * A_PART_BYTES, q[p][1], q[p][0]);
      else
        ldg256_cg(src + p * A_PART_BYTES, q[p][0], q[p][1]);
    }
  };
  if (EPI == EPI_MUL_DCELU && y_early && half < ngroups) {
    load_y(half, 0, yq[0]);
    load_y(half, 1, yq[1]);
  }
  mbar_wait(tfull_bar, tfull_parity);
  tc_fence_after();
  if (EPI == EPI_MUL_DCELU && !y_early && half < ngroups) {
    load_y(half, 0, yq[0]);
    load_y(half, 1, yq[1]);
  }

  // one 8-column chunk (c8 = 0 / 1) of half hh of group g: accumulator registers -> packed pieces wp[piece][c8 * 4 ..]
  auto chunk = [&](int g, auto hh_c, auto c8_c, const uint32_t (&r)[8], uint32_t (&wp)[PARTS][8]) {
    constexpr int hh = decltype(hh_c)::value, c8 = decltype(c8_c)::value;
    const int c0 = g * 32 + hh * 16;   // first column of this half inside the tile
#pragma unroll
    for (int i = 4 * c8; i < 4 * c8 + 4; ++i) {
      const f32x2 acc = pack2(__uint_as_float(r[2 * (i - 4 * c8)]), __uint_as_float(r[2 * (i - 4 * c8) + 1]));
      float o0, o1;
      if (EPI == EPI_MUL_DCELU) {
        uint32_t yw[PARTS];
#pragma unroll
        for (int p = 0; p < PARTS; ++p) yw[p] = u4_word(yq[hh][p][i >> 2], i & 3);
        const f32x2 y = join_pair(yw);
        float y0, y1, d0, d1;
        unpack2(y, y0, y1);
        unpack2(fma2(y, cy2, a2), d0, d1);
        d0 = y0 > 0.f ? a_s : d0;
        d1 = y1 > 0.f ? a_s : d1;
        unpack2(mul2(acc, pack2(d0, d1)), o0, o1);
      } else {
        const f32x2 x = fma2(acc, a2, *reinterpret_cast<const f32x2*>(bias + c0 + 2 * i));
        float x0, x1, t0, t1, n0, n1;
        unpack2(x, x0, x1);
        unpack2(mul2(x, kx2), t0, t1);
        const f32x2 n = fma2(al2, pack2(ex2_approx(t0), ex2_approx(t1)), nal2);
        unpack2(n, n0, n1);
        if (EPI == EPI_BIAS_CELU) {
          o0 = x0 > 0.f ? x0 : n0;
          o1 = x1 > 0.f ? x1 : n1;
        } else {  // EPI_HEAD: a = celu(x); energy += a w4; output = seed w4 celu'(a)
          const f32x2 w = *reinterpret_cast<const f32x2*>(w4 + c0 + 2 * i);
          e_acc2 = fma2(pack2(x0 > 0.f ? x0 : n0, x1 > 0.f ? x1 : n1), w, e_acc2);
          float d0, d1;
          unpack2(fma2(n, ia2, one2), d0, d1);
          d0 = x0 > 0.f ? 1.0f : d0;
          d1 = x1 > 0.f ? 1.0f : d1;
          unpack2(mul2(mul2(w, seed2), pack2(d0, d1)), o0, o1);
        }
      }
      omax = fmaxf(omax, fmaxf(fabsf(o0), fabsf(o1)));
      uint32_t w[PARTS];
      split_pair(o0, o1, w);
#pragma unroll
      for (int p = 0; p < PARTS; ++p) wp[p][i] = w[p];
    }
  };
  // after both chunks of a half: refill the stored-activation registers, store the half's sector of every piece
  auto finish = [&](int g, auto hh_c, const uint32_t (&wp)[PARTS][8]) {
    constexpr int hh = decltype(hh_c)::value;
    if (EPI == EPI_MUL_DCELU && g + 2 < ngroups) load_y(g + 2, hh, yq[hh]);
    const uint32_t sec = (uint32_t)(hh ^ (int)(sw >> 1)) << 5;
    if (g_out) {
      unsigned char* dst = ct + (size_t)g * A_BLOCK_BYTES + sec;
#pragma unroll
      for (int p = 0; p < PARTS; ++p) {
        const uint4 lo = make_uint4(wp[p][0], wp[p][1], wp[p][2], wp[p][3]);   // columns 0-7 of the half
        const uint4 hi = make_uint4(wp[p][4], wp[p][5], wp[p][6], wp[p][7]);   // columns 8-15
        if (swapped)
          stg256(dst + p * A_PART_BYTES, hi, lo);
        else
          stg256(dst + p * A_PART_BYTES, lo, hi);
      }
    }
    if (s_out) {
      const uint32_t dst = s_row + (uint32_t)g * A_BLOCK_BYTES + sec;
#pragma unroll
      for (int p = 0; p < PARTS; ++p) {
        const uint4 lo = make_uint4(wp[p][0], wp[p][1], wp[p][2], wp[p][3]);
        const uint4 hi = make_uint4(wp[p][4], wp[p][5], wp[p][6], wp[p][7]);
        sts128(dst + p * A_PART_BYTES, swapped ? hi : lo);
        sts128(dst + p * A_PART_BYTES + 16, swapped ? lo : hi);
      }
      if (hh == 1) {
        // K-block complete for this warp's 32 rows: generic-proxy writes -> visible to the tensor cores
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&res_bar[tl.n0 / TK + g]);
      }
    }
  };

  {
    // TMEM loads run one 8-column chunk ahead of the math (two statically indexed register sets)
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    uint32_t r0[8], r1[8];
    uint32_t wp[PARTS][8];   // packed 16-bit pairs of the 8 column pairs of a half, per piece
    if (half < ngroups) tmem_ld8_issue(taddr + half * 32, r0);
    for (int g = half; g < ngroups; g += 2) {
      tmem_ld_wait8(r0);
      tmem_ld8_issue(taddr + g * 32 + 8, r1);
      chunk(g, I0{}, I0{}, r0, wp);
      tmem_ld_wait8(r1);
      tmem_ld8_issue(taddr + g * 32 + 16, r0);
      chunk(g, I0{}, I1{}, r1, wp);
      finish(g, I0{}, wp);
      tmem_ld_wait8(r0);
      tmem_ld8_issue(taddr + g * 32 + 24, r1);
      chunk(g, I1{}, I0{}, r0, wp);
      tmem_ld_wait8(r1);
      if (g + 2 < ngroups) tmem_ld8_issue(taddr + (g + 2) * 32, r0);
      chunk(g, I1{}, I1{}, r1, wp);
      finish(g, I1{}, wp);
    }
  }
  if (EPI == EPI_HEAD) {
    // the two warps of a row hold the even / odd column groups: combine through shared memory
    float e0, e1;
    unpack2(e_acc2, e0, e1);
    e_part[warp * 32 + lane] = e0 + e1;
    asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");
    if (half == 0)
      args.e_member[(size_t)tl.mem * args.rows_cap + my_row] =
          row_valid ? e_part[warp * 32 + lane] + e_part[(warp + 4) * 32 + lane] + sp.b4[tl.mem] : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");
  }
}


// The same epilogue with SIXTEEN warps: the four warps of a TMEM lane quadrant split a tile by (group parity, 16-column
// half) -- warp w: quadrant w & 3, groups g = (w >> 3), (w >> 3) + 2, ..., half (w >> 2) & 1 -- so every warp does half
// of what one of the eight does above, whatever the tile width, with no barrier between warps (the round-1/2 sixteen-warp
// variant paired warps on one staging buffer): a half of a row is one 32-byte sector per piece, written / read by its
// own thread.  The point is not arithmetic throughput: a tile's epilogue is three transfers on three different paths
// -- tensor memory -> registers (64 B/clk), registers -> L2 (64 B/clk), and for the backward the stored activation
// L2 -> registers -- and eight warps with one load in flight each leave them idle most of the time.
template <int EPI>
__device__ __forceinline__ void tile_epilogue_direct16(const Args& args, const Tile& tl, const Species& sp, uint32_t taddr,
                                                       const float* __restrict__ bias, const float* __restrict__ w4,
                                                       float* e_part, int warp, int lane, uint64_t* tfull_bar,
                                                       uint32_t tfull_parity, float& omax, uint64_t* ydep_bar,
                                                       uint32_t ydep_parity) {
  static_assert(EPI == EPI_BIAS_CELU || EPI == EPI_MUL_DCELU || EPI == EPI_HEAD, "tiled-output epilogues only");
  const int quad = warp & 3, hh = (warp >> 2) & 1, gp = warp >> 3;
  const int r_tile = quad * 32 + lane;
  const uint32_t sw = (uint32_t)(lane >> 1) & 3u;
  const bool swapped = sw & 1u;
  const uint32_t row_base = (uint32_t)(r_tile >> 3) * 512u + (uint32_t)(r_tile & 7) * 64u + ((uint32_t)(hh ^ (int)(sw >> 1)) << 5);
  const bool tiled_out = EPI != EPI_HEAD || args.want_backward;
  const int my_row = tl.rt * TM + r_tile;
  unsigned char* ct = reinterpret_cast<unsigned char*>(args.C) +
                      ((size_t)tl.rt * args.c_kblocks + (size_t)(tl.mem * sp.c_moff + tl.n0) / TK) * A_BLOCK_BYTES + row_base;
  const int ngroups = tl.bn / 32;
  const float os = args.out_scale;
  const float a_s = sp.acc_scale * (EPI == EPI_HEAD ? 1.0f : os);
  const f32x2 a2 = pack2(a_s, a_s);
  const float inv_alpha = 1.0f / args.alpha;
  const float kx = (EPI == EPI_HEAD ? 1.0f : 1.0f / os) * 1.4426950408889634f * inv_alpha;
  const float al = args.alpha * (EPI == EPI_HEAD ? 1.0f : os);
  const f32x2 kx2 = pack2(kx, kx), al2 = pack2(al, al), nal2 = pack2(-al, -al);
  const float cy = inv_alpha * args.y_inv_scale * a_s;
  const f32x2 cy2 = pack2(cy, cy);
  const f32x2 ia2 = pack2(inv_alpha, inv_alpha), one2 = pack2(1.0f, 1.0f);
  float seed = 0.f;
  bool row_valid = false;
  if (EPI == EPI_HEAD) {
    row_valid = args.row_atom[my_row] >= 0;
    seed = row_valid ? args.member_scale[tl.mem] * os : 0.f;
  }
  const f32x2 seed2 = pack2(seed, seed);
  f32x2 e_acc2 = pack2(0.f, 0.f);

  uint4 yq[PARTS][2];   // stored activation of this row, this warp's half of the group in flight: [piece][chunk]
  auto load_y = [&](int g) {
    const unsigned char* src = ct + (size_t)g * A_BLOCK_BYTES;
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
      if (swapped)
        ldg256_cg(src + p * A_PART_BYTES, yq[p][1], yq[p][0]);
      else
        ldg256_cg(src + p * A_PART_BYTES, yq[p][0], yq[p][1]);
    }
  };
  if (EPI == EPI_MUL_DCELU) {
    // the producer has acquired this unit's inputs: the stored activation may be read while the main loop runs
    mbar_wait(ydep_bar, ydep_parity);
    if (gp < ngroups) load_y(gp);
  }
  mbar_wait(tfull_bar, tfull_parity);
  tc_fence_after();

  uint32_t wp[PARTS][8];
  auto chunk = [&](int g, auto c8_c, const uint32_t (&r)[8]) {
    constexpr int c8 = decltype(c8_c)::value;
    const int c0 = g * 32 + hh * 16;
#pragma unroll
    for (int i = 4 * c8; i < 4 * c8 + 4; ++i) {
      const f32x2 acc = pack2(__uint_as_float(r[2 * (i - 4 * c8)]), __uint_as_float(r[2 * (i - 4 * c8) + 1]));
      float o0, o1;
      if (EPI == EPI_MUL_DCELU) {
        uint32_t yw[PARTS];
#pragma unroll
        for (int p = 0; p < PARTS; ++p) yw[p] = u4_word(yq[p][i >> 2], i & 3);
        const f32x2 y = join_pair(yw);
        float y0, y1, d0, d1;
        unpack2(y, y0, y1);
        unpack2(fma2(y, cy2, a2), d0, d1);
        d0 = y0 > 0.f ? a_s : d0;
        d1 = y1 > 0.f ? a_s : d1;
        unpack2(mul2(acc, pack2(d0, d1)), o0, o1);
      } else {
        const f32x2 x = fma2(acc, a2, *reinterpret_cast<const f32x2*>(bias + c0 + 2 * i));
        float x0, x1, t0, t1, n0, n1;
        unpack2(x, x0, x1);
        unpack2(mul2(x, kx2), t0, t1);
        const f32x2 n = fma2(al2, pack2(ex2_approx(t0), ex2_approx(t1)), nal2);
        unpack2(n, n0, n1);
        if (EPI == EPI_BIAS_CELU) {
          o0 = x0 > 0.f ? x0 : n0;
          o1 = x1 > 0.f ? x1 : n1;
        } else {
          const f32x2 w = *reinterpret_cast<const f32x2*>(w4 + c0 + 2 * i);
          e_acc2 = fma2(pack2(x0 > 0.f ? x0 : n0, x1 > 0.f ? x1 : n1), w, e_acc2);
          float d0, d1;
          unpack2(fma2(n, ia2, one2), d0, d1);
          d0 = x0 > 0.f ? 1.0f : d0;
          d1 = x1 > 0.f ? 1.0f : d1;
          unpack2(mul2(mul2(w, seed2), pack2(d0, d1)), o0, o1);
        }
      }
      omax = fmaxf(omax, fmaxf(fabsf(o0), fabsf(o1)));
      uint32_t w[PARTS];
      split_pair(o0, o1, w);
#pragma unroll
      for (int p = 0; p < PARTS; ++p) wp[p][i] = w[p];
    }
  };
  {
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    uint32_t r0[8], r1[8];
    if (gp < ngroups) tmem_ld8_issue(taddr + gp * 32 + hh * 16, r0);
    for (int g = gp; g < ngroups; g += 2) {
      tmem_ld_wait8(r0);
      tmem_ld8_issue(taddr + g * 32 + hh * 16 + 8, r1);
      chunk(g, I0{}, r0);
      tmem_ld_wait8(r1);
      if (g + 2 < ngroups) tmem_ld8_issue(taddr + (g + 2) * 32 + hh * 16, r0);
      chunk(g, I1{}, r1);
      if (EPI == EPI_MUL_DCELU && g + 2 < ngroups) load_y(g + 2);
      if (tiled_out) {
        unsigned char* dst = ct + (size_t)g * A_BLOCK_BYTES;
#pragma unroll
        for (int p = 0; p < PARTS; ++p) {
          const uint4 lo = make_uint4(wp[p][0], wp[p][1], wp[p][2], wp[p][3]);
          const uint4 hi = make_uint4(wp[p][4], wp[p][5], wp[p][6], wp[p][7]);
          if (swapped)
            stg256(dst + p * A_PART_BYTES, hi, lo);
          else
            stg256(dst + p * A_PART_BYTES, lo, hi);
        }
      }
    }
  }
  if (EPI == EPI_HEAD) {
    float e0, e1;
    unpack2(e_acc2, e0, e1);
    e_part[warp * 32 + lane] = e0 + e1;
    asm volatile("bar.sync 1, %0;" ::"n"(16 * 32) : "memory");
    if (warp < 4)
      args.e_member[(size_t)tl.mem * args.rows_cap + my_row] =
          row_valid ? e_part[warp * 32 + lane] + e_part[(warp + 4) * 32 + lane] + e_part[(warp + 8) * 32 + lane] +
                          e_part[(warp + 12) * 32 + lane] + sp.b4[tl.mem]
                    : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(16 * 32) : "memory");
  }
}

}  // namespace tc
}  // namespace ani
