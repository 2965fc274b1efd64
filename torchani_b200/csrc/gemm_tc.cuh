// Persistent, warp-specialised, TMA-fed tcgen05 grouped GEMM for the ensemble MLP (sm_100a).
//
//   C[128-row tile, bn] = epilogue( A[128, K] x B[bn, K]^T )        both operands K-major
//
// fp32 accuracy on the tensor cores from 16-bit pieces (common.cuh, ANI_OPND_FP16X2):
//   * default "2 x fp16": every fp32 operand x is stored as two IEEE half pieces of s*x
//     (s*x = p1 + p2, residual < 2^-22 |s*x|; s = a power of two per operand class that keeps p2 a
//     normal half); the MMA thread issues three kind::f16 products per K-step,
//         a2 b1, a1 b2, a1 b1          (the dropped a2 b2 is < 2^-22 relative),
//     into one fp32 accumulator in tensor memory; the epilogue multiplies by 1/(s_a s_b) (exact).
//     4 bytes per element and half the tensor time of the alternative:
//   * "3 x bf16": x = p1 + p2 + p3 bfloat16 pieces, six products (a3b1, a1b3, a2b2, a2b1, a1b2,
//     a1b1), 6 bytes per element, no scale.
// The six launches of a step are bound by the bytes they move through the L2, not by the MMAs
// (DESIGN.md 4.1), so bytes per element is the figure of merit.
//
// BOTH operands live in global memory in the "tiled operand" layout of include/ani_b200.h:
// 32-column K-blocks, [p1 rows x 64 B | p2 rows x 64 B (| p3 rows x 64 B)], every 8-row group in
// SWIZZLE_64B order.
//   * B (weights) is tiled once at model-pack time,
//   * A (activations / gradients) is written in that layout by the epilogue of the GEMM (or by
//     the AEV kernel) that produces it.
// A K-block of a tile is therefore ONE contiguous byte range that one thread moves with
// cp.async.bulk (TMA) straight into the shared-memory layout the MMA descriptors expect; no
// thread ever touches operand data.
//
// Roles (10 warps, one CTA per SM, persistent over the device-side tile list):
//   warps 0-7  epilogue : tcgen05.ld (thread = row; warps w and w+4 share TMEM lanes and take
//                         alternate 32-column groups), bias + CELU | * CELU'(stored activation) |
//                         final layer + gradient seed | plain; split into pieces, staged in shared
//                         memory in the final byte order and written by TMA bulk stores
//   warp  8    MMA      : TMEM alloc, one lane issues tcgen05.mma / tcgen05.commit
//   warp  9    producer : one lane arms the mbarrier (expect_tx) and issues the bulk copies
// Pipelines: smem full/empty (2-6 stages of PARTS x (8 KB + bn x 64 B), sized on the device from the
// widest accumulator of the launch) and TMEM full/empty (2 x 256 columns), so the epilogue of
// tile i overlaps the main loop of tile i+1; TMEM loads run one half group ahead of the math.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"

namespace ani {
namespace tc {

constexpr int TM = ANI_TILE_ROWS;        // 128 rows per tile == UMMA M
constexpr int TN_MAX = 256;              // UMMA N (columns of one accumulator)
constexpr int TK = OPND_KB;              // 32 columns per K-block = one 64-byte swizzle row of 16-bit pieces
constexpr int ROW_BYTES = OPND_ROW_BYTES;        // 64
constexpr int GROUP_BYTES = 8 * ROW_BYTES;       // 8-row swizzle group = 512 B (descriptor SBO)
constexpr int PARTS = OPND_PARTS;                // 2 (fp16) or 3 (bf16)
constexpr int MAX_STAGES = 6;
constexpr int A_PART_BYTES = OPND_PART_BYTES;    // 8 KB (one piece of one A K-block)
constexpr int A_BLOCK_BYTES = OPND_BLOCK_BYTES;  // 16 / 24 KB: [p1 | p2 (| p3)], contiguous in global memory
constexpr int EPI_PART_BYTES = 32 * ROW_BYTES;   // one piece of a warp's 32 rows x 32 columns = 2 KB
constexpr int EPI_STAGE_BYTES = PARTS * EPI_PART_BYTES;  // 4 / 6 KB per epilogue warp and buffer
constexpr int NUM_EPI_WARPS = 8, MMA_WARP = 8, PROD_WARP = 9;
// always (almost) the whole SM: the pipeline depth adapts on the device.  6 KB of the 227 KB are
// left for the static shared memory (tile map, barriers, bias staging, EPI_HEAD partial sums)
constexpr int SMEM_BYTES = 227 * 1024 - 6144;
constexpr int THREADS = (NUM_EPI_WARPS + 2) * 32;  // 320
constexpr int TMEM_COLS = 512;

enum { EPI_BIAS_CELU = 0, EPI_MUL_DCELU = 1, EPI_PLAIN = 2, EPI_HEAD = 3 };

struct Species {
  const unsigned char* Bt;  // tiled B operand
  const float* bias;  // [N] (+ member * bias_mstride) or nullptr
  int K, N;
  int a_moff, c_moff, bias_mstride;  // per-member column offsets into A / C (multiples of 32)
  const float* w4;    // EPI_HEAD: final layer weights [M][N] and biases [M]
  const float* b4;
  // split-K over the members (layer-1 backward): all members share ONE B operand with b_kblocks
  // K-blocks, member m starts at K-block m * b_kb_moff.  0: one B operand per member.
  int b_kblocks, b_kb_moff;
  float acc_scale;  // 1 / (scale of A x scale of this B operand): multiplies the raw accumulator
};

struct Args {
  const unsigned char* A;       // tiled activation matrix [row tile][a_kblocks][p1 | p2 (| p3)]
  void* C;                      // tiled activation matrix (EPI_PLAIN: plain row-major float [rows][ldc])
  int a_kblocks, c_kblocks;     // 32-column blocks per row of A / C  (= leading dimension / 32)
  int ldc;                      // EPI_PLAIN only
  int members;                  // GEMMs per row tile
  const int32_t* layout_info;   // [4 + S + 1]: ..., first row tile of species s, total row tiles
  const int32_t* kblocks;       // optional list of live 32-wide K-blocks: [count, ids...]  (layer-1 forward)
  const int32_t* nblocks;       // optional list of live 32-wide column blocks of C          (layer-1 backward)
  int num_species;
  float alpha;
  // EPI_HEAD (layer 3 + final layer + gradient seed fused in the epilogue)
  float* e_member;              // [M][rows_cap]
  const int32_t* row_atom;      // [rows_cap], -1 for padding rows
  int rows_cap;
  int want_backward;
  int c_accumulate;             // EPI_PLAIN: C += tile (vector RED), C zeroed by the caller
  long long* trace;             // optional clock64 stamps [cta < 4][tile < 8][role 3][4] (ani_b200_debug_gemm_trace)
  float out_scale;              // operand scale of a tiled C (OPND_SCALE_VALUE activations / OPND_SCALE_GRAD gradients)
  float y_inv_scale;            // EPI_MUL_DCELU: 1 / scale of the stored activation that C overwrites
  int32_t* status;              // ANI_STATUS_OPERAND_RANGE is raised here (may be NULL)
  int allow_narrow;             // short tile lists may split every accumulator into two column tiles (not EPI_HEAD)
  int win_idx, win_cnt;         // this launch covers window win_idx of win_cnt equal parts of every species' row tiles
                                // (mlp.cu: a step may run as several launches whose working sets stay in the L2)
  int epi_direct;               // tiled outputs straight from registers (gemm_epilogue.cuh); 0: shared-memory staging + TMA stores
  int b_compact;                // with `nblocks`: B holds ONLY the live column blocks, packed like a dense operand of
                                // nb_count * 32 rows (mlp.cu: k_zero_live_blocks builds it every step) -- one bulk copy
                                // per K-block instead of one 2 KB copy per live block and piece
  int debug;                    // timing experiments only (ANI_B200_GEMM_DEBUG): 2 no copies, 4 no MMA, 8 no epilogue
  float member_scale[ANI_MAX_MEMBERS];
  Species sp[ANI_MAX_SPECIES];
};

// ---- PTX wrappers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared, completion signalled on the mbarrier (complete_tx::bytes)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// TMA bulk store shared -> global (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void red_add_v4(float* dst, const float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (half or bf16 inputs per the instruction
// descriptor, fp32 accumulate), single CTA
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ---- CTA pairs (cta_group::2): two CTAs of a cluster work on a 256-row tile; each loads its own 128
// rows of A and HALF of B, the tensor cores of both SMs read both halves; one thread of the leader
// (cluster rank 0) issues the MMAs and signals the barriers of both CTAs
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// wait with cluster-scope acquire (the arrivals come from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP_C:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE_C;\n\t"
      "bra.uni WAIT_LOOP_C;\n\t"
      "WAIT_DONE_C:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all MMAs issued so far -> one arrival on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const unsigned short mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 16 consecutive accumulator columns of this thread's TMEM lane: asynchronous issue ...
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
// ... and the wait; the registers are threaded through the asm so no use can be scheduled above it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// shared-memory matrix descriptor: K-major, SWIZZLE_64B, 8-row groups 512 B apart
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);   // start address
  d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(GROUP_BYTES >> 4) << 32;       // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
  d |= (uint64_t)4 << 61;                        // SWIZZLE_64B
  return d;
}
// instruction descriptor: D=f32, A=B=f16 (format 0) or bf16 (format 1), both K-major, M=128, N=bn
__device__ __forceinline__ uint32_t make_idesc(int bn, int m = TM) {
  constexpr uint32_t fmt = ANI_OPND_FP16X2 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// CELU(x) = max(0,x) + min(0, alpha*(exp(x/alpha)-1)) with exp via ex2.approx (rel. error ~2^-22:
// the negative branch is bounded by alpha, so the absolute error is < 1e-8 for alpha = 0.1)
struct CeluConst {
  float alpha, inv_alpha, inv_alpha_log2e;
};
__device__ __forceinline__ float celu(float x, const CeluConst& c) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * c.inv_alpha_log2e));
  return x > 0.f ? x : fmaf(c.alpha, e, -c.alpha);
}
__device__ __forceinline__ float dcelu_from_out(float y, const CeluConst& c) {
  return y > 0.f ? 1.0f : fmaf(y, c.inv_alpha, 1.0f);
}

// ---- tile enumeration -----------------------------------------------------------------------
// Row tiles of one species are contiguous; tile t -> (species, row tile, member, n0, bn).
constexpr int MAX_BLOCKS = 64;         // ldx / 32 <= 64
struct TileMap {
  int first_rt[ANI_MAX_SPECIES + 1];   // first row tile of each species inside this launch's window
  int cnt_rt[ANI_MAX_SPECIES];         // row tiles of each species inside the window
  int ntn[ANI_MAX_SPECIES];            // N tiles per (row tile, member)
  int prefix[ANI_MAX_SPECIES + 1];     // exclusive prefix of tile counts
  int n_eff[ANI_MAX_SPECIES];          // columns actually computed (compacted when nblocks is given)
  int tn[ANI_MAX_SPECIES];             // columns per tile: TN_MAX, or half an accumulator for short lists
  int kb_count, nb_count;              // live K-blocks (-1: dense) / live column blocks (-1: dense)
  int kb[MAX_BLOCKS], nb[MAX_BLOCKS];
  int stages, stage_bytes, epi_bufs;   // shared-memory budget of this launch
};

struct Tile {
  int s, rt, mem, n0, bn;
  int rt_last;  // last row tile of the species (a CTA pair may own one row tile too many)
};

// pair: the unit of work is a PAIR of row tiles (rank r of the cluster takes row tile rt + r)
__device__ __forceinline__ void build_tile_map(const Args& a, TileMap& tm, bool pair = false) {
  const int S = a.num_species;
  int run = 0;
  tm.kb_count = tm.nb_count = -1;
  if (a.kblocks) {
    tm.kb_count = min(a.kblocks[0], MAX_BLOCKS);
    for (int i = 0; i < tm.kb_count; ++i) tm.kb[i] = a.kblocks[1 + i];
  }
  if (a.nblocks) {
    tm.nb_count = min(a.nblocks[0], MAX_BLOCKS);
    for (int i = 0; i < tm.nb_count; ++i) tm.nb[i] = a.nblocks[1 + i];
  }
  const int wc = a.win_cnt > 1 ? a.win_cnt : 1, wi = a.win_cnt > 1 ? a.win_idx : 0;
  for (int s = 0; s < S; ++s) {
    const int f = a.layout_info[4 + s], nrt_all = a.layout_info[4 + s + 1] - f;
    const int lo = f + (int)((long long)nrt_all * wi / wc), hi = f + (int)((long long)nrt_all * (wi + 1) / wc);
    tm.first_rt[s] = lo;
    tm.cnt_rt[s] = hi - lo;
    tm.n_eff[s] = tm.nb_count >= 0 ? tm.nb_count * 32 : a.sp[s].N;
    tm.tn[s] = TN_MAX;
    tm.ntn[s] = (tm.n_eff[s] + TN_MAX - 1) / TN_MAX;
  }
  tm.first_rt[S] = a.layout_info[4 + S];
  auto count = [&]() {
    int run = 0;
    for (int s = 0; s < S; ++s) {
      tm.prefix[s] = run;
      const int nrt = tm.cnt_rt[s];
      run += (pair ? (nrt + 1) / 2 : nrt) * a.members * tm.ntn[s];
    }
    tm.prefix[S] = run;
    return run;
  };
  const int wide = count();
  // Short lists (less than half a wave of 256-column tiles: 1 k-atom systems, multi-GPU shards): split every
  // accumulator into two column tiles -- twice the CTAs at work, each with half the main loop and half the epilogue,
  // which is what the latency of the layer chain is made of.  (Tiles never straddle a packed 256-row B tile.)
  if (a.allow_narrow && !pair && wide > 0 && 2 * wide <= (int)gridDim.x) {
    for (int s = 0; s < S; ++s) {
      tm.tn[s] = tm.n_eff[s] > TN_MAX ? TN_MAX / 2 : max(32, ((tm.n_eff[s] / 32 + 1) / 2) * 32);
      tm.ntn[s] = (tm.n_eff[s] + tm.tn[s] - 1) / tm.tn[s];
    }
    count();
  }
  int bn_max = 32;
  for (int s = 0; s < S; ++s)
    if (tm.cnt_rt[s] > 0) bn_max = max(bn_max, min(tm.tn[s], tm.n_eff[s]));
  tm.stage_bytes = A_BLOCK_BYTES + PARTS * (pair ? bn_max / 2 : bn_max) * ROW_BYTES;  // a pair member holds half of B
  // two store-staging buffers per epilogue warp if that still leaves a double-buffered main loop
  const int avail = SMEM_BYTES - 1024;
  tm.epi_bufs = a.epi_direct ? 0 : (avail - 2 * NUM_EPI_WARPS * EPI_STAGE_BYTES) / tm.stage_bytes >= 2 ? 2 : 1;
  // (a single store buffer per warp would buy one more main-loop stage: measured on B200, no gain --
  // 0.2374 vs 0.2358 ms for the six launches)
  tm.stages = min(MAX_STAGES, (avail - tm.epi_bufs * NUM_EPI_WARPS * EPI_STAGE_BYTES) / tm.stage_bytes);
}

__device__ __forceinline__ Tile decode_tile(const Args& a, const TileMap& tm, int t, bool pair = false) {
  Tile x;
  int s = 0;
  while (t >= tm.prefix[s + 1]) ++s;
  const int local = t - tm.prefix[s];
  const int ntn = tm.ntn[s];
  const int nt = local % ntn;
  const int rm = local / ntn;
  x.s = s;
  x.mem = rm % a.members;
  x.rt = tm.first_rt[s] + (pair ? 2 : 1) * (rm / a.members);
  x.rt_last = tm.first_rt[s] + tm.cnt_rt[s] - 1;
  x.n0 = nt * tm.tn[s];
  x.bn = min(tm.tn[s], tm.n_eff[s] - x.n0);
  return x;
}

// ---- split of two adjacent (already scaled) fp32 values into PARTS packed 16-bit pairs (low half = a)
__device__ __forceinline__ void split_pair(float a, float b, uint32_t (&w)[PARTS]) {
#if ANI_OPND_FP16X2
  __half2 h = __floats2half2_rn(a, b);
  w[0] = *reinterpret_cast<uint32_t*>(&h);
  const float2 f = __half22float2(h);
  h = __floats2half2_rn(a - f.x, b - f.y);
  w[1] = *reinterpret_cast<uint32_t*>(&h);
#else
#pragma unroll
  for (int p = 0; p < PARTS; ++p) {
    __nv_bfloat162 q = __floats2bfloat162_rn(a, b);
    w[p] = *reinterpret_cast<uint32_t*>(&q);
    a -= __uint_as_float(w[p] << 16);
    b -= __uint_as_float(w[p] & 0xffff0000u);
  }
#endif
}
// sum of the pieces of 8 consecutive columns (one 16-byte chunk per piece; q[2 * p]) -> 8 floats
// (still multiplied by the operand scale)
__device__ __forceinline__ void join_chunk(const uint4* q, float* y) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float lo = 0.f, hi = 0.f;
#pragma unroll
    for (int p = PARTS - 1; p >= 0; --p) {  // smallest piece first
      const uint4& v = q[2 * p];
      const uint32_t word = i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
#if ANI_OPND_FP16X2
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&word));
      lo += f.x;
      hi += f.y;
#else
      lo += __uint_as_float(word << 16);
      hi += __uint_as_float(word & 0xffff0000u);
#endif
    }
    y[2 * i] = lo;
    y[2 * i + 1] = hi;
  }
}

template <int EPI>
__device__ __forceinline__ void tile_epilogue_direct(const Args& args, const Tile& tl, int rt_mine, const Species& sp,
                                                     uint32_t taddr, const float* __restrict__ bias,
                                                     const float* __restrict__ w4, float* e_part, int warp, int lane,
                                                     uint64_t* tfull_bar, uint32_t tfull_parity, float& omax, bool y_early,
                                                     unsigned char* res = nullptr, uint64_t* res_bar = nullptr,
                                                     bool c_store = true);

// ---- the kernel -----------------------------------------------------------------------------
template <int EPI, bool PAIR = false>
__global__ void __launch_bounds__(THREADS, 1) k_gemm_tc(const __grid_constant__ Args args) {
  extern __shared__ unsigned char smem_raw[];
  // 1024-byte aligned operand tiles (swizzle groups are 8 rows x 64 B)
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ TileMap tm;
  __shared__ float e_part[NUM_EPI_WARPS * 32];  // EPI_HEAD: partial row energies of the two column halves
  __shared__ __align__(16) float s_bias[2][TN_MAX];  // bias (and final-layer weights) of the tile in flight,
  __shared__ __align__(16) float s_w4[2][TN_MAX];    // double-buffered by tile parity
  auto stamp = [&](int tile_local, int role, int slot) {
    if (args.trace && blockIdx.x < 4 && tile_local < 8)
      args.trace[(((size_t)blockIdx.x * 8 + tile_local) * 3 + role) * 4 + slot] = clock64();
  };
  if (threadIdx.x == 0) build_tile_map(args, tm, PAIR);
  __syncthreads();
  // CTA pair: cluster of two consecutive CTAs; both walk the same list of row-tile pairs
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int unit_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int STAGES = tm.stages, STAGE_BYTES = tm.stage_bytes, EPI_BUFS = tm.epi_bufs;
  unsigned char* epi_stage = smem + STAGES * STAGE_BYTES;  // 8 warps x EPI_BUFS x 6 KB store staging
  __shared__ __align__(8) uint64_t bars[2 * MAX_STAGES + 5];
  uint64_t* full = bars;                         // [STAGES]  TMA bytes -> MMA
  uint64_t* empty = bars + MAX_STAGES;           // [STAGES]  MMA (commit) -> producer
  uint64_t* tfull = bars + 2 * MAX_STAGES;       // [2]       MMA (commit) -> epilogue
  uint64_t* tempty = bars + 2 * MAX_STAGES + 2;  // [2]       epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 4);
  __shared__ uint64_t pfull[MAX_STAGES];         // pair mode, leader: "the peer's operands of this stage have landed"

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);   // the expect_tx arrival of the producer lane (+ the transaction bytes)
      mbar_init(&empty[i], 1);
      mbar_init(&pfull[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      // one elected arrival per epilogue warp; in pair mode the leader also counts the peer's warps
      mbar_init(&tempty[i], PAIR ? 2 * NUM_EPI_WARPS : NUM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (PAIR) cluster_sync_all();  // the peer's barriers exist before anything is signalled across
  if (warp == MMA_WARP) {
    if (PAIR)
      tmem_alloc2(tmem_slot, TMEM_COLS);
    else
      tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  if (PAIR)
    cluster_sync_all();
  else
    __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // programmatic dependent launch: the next kernel of the stream may start scheduling its CTAs from
  // here on (they find room when CTAs of this grid exit); everything above did not touch data the
  // previous kernel writes (layout_info / block lists are older), everything below may: wait for
  // the previous grid to complete and flush.  Both are no-ops in a plain launch.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int total_tiles = tm.prefix[args.num_species];
  // K-blocks are 32 columns, the same granularity as the optional live-block lists
  auto num_kb = [&](int K) { return tm.kb_count >= 0 ? tm.kb_count : (K + TK - 1) / TK; };
  auto kb_id = [&](int i) { return tm.kb_count >= 0 ? tm.kb[i] : i; };

  if (warp == PROD_WARP) {
    // ================================ producer (TMA) ================================
    uint32_t stage = 0, phase = 0;
    int tloc = 0;
    for (int t = unit0; t < total_tiles; t += unit_stride, ++tloc) {
      const Tile tl = decode_tile(args, tm, t, PAIR);
      const Species& sp = args.sp[tl.s];
      const int nkb = num_kb(sp.K);
      const int rt_mine = min(tl.rt + (int)rank, tl.rt_last);  // odd species: the last pair has one real row tile
      if (lane == 0) stamp(tloc, 0, 0);
      const int nkb_all = sp.b_kb_moff ? sp.b_kblocks : (sp.K + TK - 1) / TK;  // K-blocks of the stored B operand
      const int kb_boff = tl.mem * sp.b_kb_moff;                               // split-K: this member's first K-block
      // A: [row tile][32-column block][p1 | p2 | p3]; this GEMM starts at column member * a_moff
      const unsigned char* At =
          args.A + ((size_t)rt_mine * args.a_kblocks + (size_t)(tl.mem * sp.a_moff) / TK) * A_BLOCK_BYTES;
      // B: [member][n tile][k block][p1 bn x 64 B | p2 | p3]
      const unsigned char* Bm =
          sp.Bt + (sp.b_kb_moff ? (size_t)0 : (size_t)tl.mem * sp.N * nkb_all * (PARTS * ROW_BYTES));
      // one piece of this CTA's B rows: all bn rows, or half of them in a CTA pair
      const uint32_t b_bytes = (uint32_t)(PAIR ? tl.bn / 2 : tl.bn) * ROW_BYTES;
      const bool dense = tm.nb_count < 0 || args.b_compact;
      // the packed B tile this one lies in
      const int n0p = tl.n0 / TN_MAX * TN_MAX, bnp = min(TN_MAX, (args.b_compact ? tm.n_eff[tl.s] : sp.N) - n0p);
      // gathered column blocks (layer-1 backward): lane -> (live block q, piece)
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
        mbar_wait(&empty[stage], phase ^ 1);
        unsigned char* st = smem + stage * STAGE_BYTES;
        const int kbi = kb_id(kb);
        const int kbb = kbi + kb_boff;
        if (!(args.debug & 2)) {
          if (lane == 0) {
            mbar_arrive_expect_tx(&full[stage], A_BLOCK_BYTES + PARTS * b_bytes);
            bulk_g2s(st, At + (size_t)kbi * A_BLOCK_BYTES, A_BLOCK_BYTES, &full[stage]);
            if (dense) {
              const unsigned char* bsrc = Bm + ((size_t)tl.n0 * nkb_all + (size_t)kbb * tl.bn) * (PARTS * ROW_BYTES);
              if (!PAIR && tl.bn == bnp) {  // the pieces are adjacent in global memory and in shared memory: one copy
                bulk_g2s(st + A_BLOCK_BYTES, bsrc, PARTS * b_bytes, &full[stage]);
              } else if (!PAIR) {           // a column tile inside a packed 256-row B tile: one copy per piece
#pragma unroll
                for (int p = 0; p < PARTS; ++p)
                  bulk_g2s(st + A_BLOCK_BYTES + p * b_bytes,
                           Bm + ((size_t)n0p * nkb_all + (size_t)kbb * bnp) * (PARTS * ROW_BYTES) +
                               (size_t)p * bnp * ROW_BYTES + (size_t)(tl.n0 - n0p) * ROW_BYTES,
                           b_bytes, &full[stage]);
              } else {      // this CTA's half of the rows of every piece
#pragma unroll
                for (int p = 0; p < PARTS; ++p)
                  bulk_g2s(st + A_BLOCK_BYTES + p * b_bytes, bsrc + (size_t)p * tl.bn * ROW_BYTES + (size_t)rank * b_bytes,
                           b_bytes, &full[stage]);
              }
            }
          }
          __syncwarp();
          if (g_active)
            bulk_g2s(st + A_BLOCK_BYTES + gpart * b_bytes + gq * 32 * ROW_BYTES,
                     Bm + g_src + (size_t)kbb * g_bns * (PARTS * ROW_BYTES), 32 * ROW_BYTES, &full[stage]);
        } else if (lane == 0) {
          mbar_arrive(&full[stage]);
        }
        __syncwarp();
        if (lane == 0 && kb == 0) stamp(tloc, 0, 1);
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (lane == 0) stamp(tloc, 0, 2);
    }
  } else if (warp == MMA_WARP) {
    // ================================ MMA issuer ================================
    uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
    int tloc = 0;
    if (PAIR && rank != 0) {
      // peer of a CTA pair: no MMAs to issue (the leader's instructions drive both tensor cores); relay
      // "my operands of this stage have landed" to the leader
      for (int t = unit0; t < total_tiles; t += unit_stride) {
        const Tile tl = decode_tile(args, tm, t, PAIR);
        const int nkb = num_kb(args.sp[tl.s].K);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);
          if (lane == 0) mbar_arrive_remote(&pfull[stage], 0);
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    } else {
      for (int t = unit0; t < total_tiles; t += unit_stride, ++tloc) {
        const Tile tl = decode_tile(args, tm, t, PAIR);
        const int nkb = num_kb(args.sp[tl.s].K);
        const uint32_t idesc = make_idesc(tl.bn, PAIR ? 2 * TM : TM);
        const uint32_t b_bytes = (uint32_t)(PAIR ? tl.bn / 2 : tl.bn) * ROW_BYTES;
        if (lane == 0) stamp(tloc, 1, 0);
        // the epilogue (of both CTAs in a pair) has drained this accumulator
        if (PAIR)
          mbar_wait_cluster(&tempty[acc], acc_phase ^ 1);
        else
          mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        if (lane == 0) stamp(tloc, 1, 1);
        const uint32_t d_tmem = tmem_base + acc * TN_MAX;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);
          if (PAIR) mbar_wait_cluster(&pfull[stage], phase);
          tc_fence_after();
          if (lane == 0 && kb == 0) stamp(tloc, 1, 2);
          if (lane == 0) {
            const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
            const uint32_t sb = sa + A_BLOCK_BYTES;
            const uint64_t a1 = make_desc(sa), a2 = make_desc(sa + A_PART_BYTES);
            const uint64_t b1 = make_desc(sb), b2 = make_desc(sb + b_bytes);
#if !ANI_OPND_FP16X2
            const uint64_t a3 = make_desc(sa + 2 * A_PART_BYTES), b3 = make_desc(sb + 2 * b_bytes);
#endif
            auto mma = [&](uint64_t da, uint64_t db, uint32_t accumulate) {
              if (PAIR)
                umma_f16_pair(d_tmem, da, db, idesc, accumulate);
              else
                umma_f16(d_tmem, da, db, idesc, accumulate);
            };
#pragma unroll
            for (int k = 0; k < TK / 16; ++k) {
              if (args.debug & 4) break;
              const uint64_t adv = (uint64_t)(k * 2);  // 16 pieces = 32 B = 2 x 16 B along the swizzle row
              // smallest terms first
#if ANI_OPND_FP16X2
              mma(a2 + adv, b1 + adv, (kb | k) != 0);
              mma(a1 + adv, b2 + adv, 1);
              mma(a1 + adv, b1 + adv, 1);
#else
              mma(a3 + adv, b1 + adv, (kb | k) != 0);
              mma(a1 + adv, b3 + adv, 1);
              mma(a2 + adv, b2 + adv, 1);
              mma(a2 + adv, b1 + adv, 1);
              mma(a1 + adv, b2 + adv, 1);
              mma(a1 + adv, b1 + adv, 1);
#endif
            }
            // smem slot free once these MMAs retire (in both CTAs of a pair)
            if (PAIR)
              umma_commit_pair(&empty[stage]);
            else
              umma_commit(&empty[stage]);
            if (kb == nkb - 1) {  // accumulator complete
              if (PAIR)
                umma_commit_pair(&tfull[acc]);
              else
                umma_commit(&tfull[acc]);
              stamp(tloc, 1, 3);
            }
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ================================ epilogue ================================
    // Thread = accumulator row (TMEM lane).  Warps w and w+4 share the 32 lanes of quadrant w & 3
    // and take alternate 32-column groups (= K-blocks of the next GEMM), each as two 16-column halves.
    uint32_t acc = 0, acc_phase = 0, buf = 0;
    float omax = 0.f;  // largest |scaled value| this thread handed to the half-precision split
    const CeluConst cc{args.alpha, 1.0f / args.alpha, 1.4426950408889634f / args.alpha};
    const int quad = warp & 3, half = warp >> 2;
    const int r_tile = quad * 32 + lane;  // row inside the 128-row tile
    uint32_t my_off[4], st_off[4];
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      my_off[ch] = swz_off(r_tile, ch);   // inside a 128-row piece (global)
      st_off[ch] = swz_off(lane, ch);     // inside this warp's 32-row staging image (shared)
    }
    // The warp's 32 rows x 64 B of one 32-column group are a contiguous 2 KB range of the tiled
    // layout per piece (pieces 8 KB apart): stage them in shared memory in that very byte order and
    // let the TMA write them (full lines, no partial-sector stores).
    unsigned char* sb0 = epi_stage + warp * (EPI_BUFS * EPI_STAGE_BYTES);
    const bool tiled_out = EPI != EPI_PLAIN && (EPI != EPI_HEAD || args.want_backward) && !(args.debug & 32);
    int tloc = 0;
    for (int t = unit0; t < total_tiles; t += unit_stride, ++tloc) {
      const Tile tl = decode_tile(args, tm, t, PAIR);
      const Species& sp = args.sp[tl.s];
      const float acc_scale = sp.acc_scale;
      // CTA pair: rank r owns row tile rt + r; the last pair of a species with an odd number of row
      // tiles has a second member without rows (it fed a copy of the last tile to the MMAs): no output
      const int rt_mine = min(tl.rt + (int)rank, tl.rt_last);
      const bool valid = !PAIR || tl.rt + (int)rank <= tl.rt_last;
      if (threadIdx.x == 0) stamp(tloc, 2, 0);
      // bias (and final-layer weights) of this tile -> shared memory while the main loop runs
      const float* __restrict__ bias = s_bias[acc];
      const float* __restrict__ w4 = s_w4[acc];
      if (EPI == EPI_BIAS_CELU || EPI == EPI_HEAD) {
        const int c = threadIdx.x;  // 256 epilogue threads == TN_MAX columns
        if (c < tl.bn) {
          // (the register-direct epilogue folds the output scale into the staged bias)
          s_bias[acc][c] = sp.bias[(size_t)tl.mem * sp.bias_mstride + tl.n0 + c] *
                           (args.epi_direct && EPI == EPI_BIAS_CELU ? args.out_scale : 1.0f);
          if (EPI == EPI_HEAD) s_w4[acc][c] = sp.w4[(size_t)tl.mem * sp.N + c];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");  // epilogue warps only
      }
      if (EPI != EPI_PLAIN && args.epi_direct && valid && !(args.debug & 8)) {
        if (threadIdx.x == 0) stamp(tloc, 2, 1);
        tile_epilogue_direct<EPI == EPI_PLAIN ? EPI_BIAS_CELU : EPI>(
            args, tl, rt_mine, sp, tmem_base + ((uint32_t)(quad * 32) << 16) + acc * TN_MAX, bias, w4, e_part, warp, lane,
            &tfull[acc], acc_phase, omax, true);
      } else if (valid) {
      const int my_row = rt_mine * TM + r_tile;
      float e_acc = 0.f, seed = 0.f;
      bool row_valid = false;
      if (EPI == EPI_HEAD) {
        row_valid = args.row_atom[my_row] >= 0;
        seed = row_valid ? args.member_scale[tl.mem] : 0.f;
      }
      // tiled C: the block of 32-column group g is [row tile][(member*c_moff + n0)/32 + g]
      unsigned char* ct = reinterpret_cast<unsigned char*>(args.C) +
                          ((size_t)rt_mine * args.c_kblocks + (size_t)(tl.mem * sp.c_moff + tl.n0) / TK) * A_BLOCK_BYTES;
      float* cplain = reinterpret_cast<float*>(args.C) + (size_t)my_row * args.ldc + (size_t)tl.mem * sp.c_moff;
      const int ngroups = tl.bn / 32;
      // stored activation (all pieces) of 16 columns = chunks 2*hh, 2*hh+1 of group g, this thread's row
      // one register set per 16-column half, refilled for the same half of the warp's next group as soon as it has
      // been consumed: the loads run a whole 32-column group of epilogue math ahead of their use
      uint4 yq[2][2 * PARTS];
      auto load_y = [&](int g, int hh, uint4 (&q)[2 * PARTS]) {
        const unsigned char* blk = ct + (size_t)g * A_BLOCK_BYTES;
#pragma unroll
        for (int p = 0; p < PARTS; ++p) {
          q[2 * p] = *reinterpret_cast<const uint4*>(blk + p * A_PART_BYTES + my_off[2 * hh]);
          q[2 * p + 1] = *reinterpret_cast<const uint4*>(blk + p * A_PART_BYTES + my_off[2 * hh + 1]);
        }
      };
      if (EPI == EPI_MUL_DCELU && half < ngroups && !(args.debug & 128)) {  // overlaps the wait for the accumulator
        load_y(half, 0, yq[0]);
        load_y(half, 1, yq[1]);
      }
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      if (threadIdx.x == 0) stamp(tloc, 2, 1);
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * TN_MAX;

      // one 16-column half of group g: raw accumulator registers -> epilogue math -> staging / store
      auto process = [&](int g, auto hh_c, const uint32_t (&r)[16]) {
        constexpr int hh = decltype(hh_c)::value;
        float y[16];
        if (EPI == EPI_MUL_DCELU) {
          join_chunk(yq[hh], y);
          join_chunk(yq[hh] + 1, y + 8);
          if (!(args.debug & 128) && g + 2 < ngroups) load_y(g + 2, hh, yq[hh]);
        }
        unsigned char* sb = sb0 + buf * EPI_STAGE_BYTES;
        if (tiled_out && hh == 0) {
          // this buffer was handed to the TMA EPI_BUFS groups ago: its read must be complete
          if (lane == 0) {
            if (EPI_BUFS == 2)
              bulk_wait_read<1>();
            else
              bulk_wait_read<0>();
          }
          __syncwarp();
        }
        const int c0 = g * 32 + hh * 16;  // first column of this half inside the tile
        float o[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float v = __uint_as_float(r[j]) * acc_scale;
          if (EPI == EPI_BIAS_CELU) {
            v = celu(v + bias[c0 + j], cc);
          } else if (EPI == EPI_MUL_DCELU) {
            v *= dcelu_from_out(y[j] * args.y_inv_scale, cc);
          } else if (EPI == EPI_HEAD) {
            const float w = w4[c0 + j];
            const float a = celu(v + bias[c0 + j], cc);
            e_acc = fmaf(a, w, e_acc);
            v = seed * w * dcelu_from_out(a, cc);
          }
          if (EPI != EPI_PLAIN) {
            v *= args.out_scale;
            omax = fmaxf(omax, fabsf(v));
          }
          o[j] = v;
        }
        if (args.debug & 32) return;
        if (EPI == EPI_PLAIN) {
          // compacted column blocks map back to their place: group g is live block n0/32 + g
          const int col = (tm.nb_count >= 0 ? tm.nb[tl.n0 / 32 + g] * 32 : tl.n0 + g * 32) + hh * 16;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 v4 = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
            if (args.c_accumulate)
              red_add_v4(cplain + col + 4 * q, v4);
            else
              *reinterpret_cast<float4*>(cplain + col + 4 * q) = v4;
          }
        } else if (tiled_out) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {  // chunk 2*hh + c = columns 8c .. 8c+7 of this half
            uint32_t w[4][PARTS];
#pragma unroll
            for (int i = 0; i < 4; ++i) split_pair(o[8 * c + 2 * i], o[8 * c + 2 * i + 1], w[i]);
            const uint32_t off = st_off[2 * hh + c];
#pragma unroll
            for (int p = 0; p < PARTS; ++p)
              *reinterpret_cast<uint4*>(sb + p * EPI_PART_BYTES + off) = make_uint4(w[0][p], w[1][p], w[2][p], w[3][p]);
          }
          if (hh == 1) {
            unsigned char* blk = ct + (size_t)g * A_BLOCK_BYTES + quad * EPI_PART_BYTES;
            fence_proxy_async();  // generic-proxy smem writes -> visible to the TMA
            __syncwarp();
            if (lane == 0) {
#pragma unroll
              for (int p = 0; p < PARTS; ++p) bulk_s2g(blk + p * A_PART_BYTES, sb + p * EPI_PART_BYTES, EPI_PART_BYTES);
              bulk_commit();
            }
            if (EPI_BUFS == 2) buf ^= 1;
          }
        }
      };

      // TMEM loads run one half group ahead of the math (two statically indexed register sets)
      if (!(args.debug & 8)) {
        uint32_t r0[16], r1[16];
        if (half < ngroups) tmem_ld16_issue(taddr + half * 32, r0);
        for (int g = half; g < ngroups; g += 2) {
          tmem_ld_wait(r0);
          tmem_ld16_issue(taddr + g * 32 + 16, r1);
          process(g, std::integral_constant<int, 0>{}, r0);
          tmem_ld_wait(r1);
          if (g + 2 < ngroups) tmem_ld16_issue(taddr + (g + 2) * 32, r0);
          process(g, std::integral_constant<int, 1>{}, r1);
        }
      }
      if (EPI == EPI_HEAD) {
        // the two warps of a row hold the even / odd column groups: combine through shared memory
        e_part[warp * 32 + lane] = e_acc;
        asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");  // epilogue warps only
        if (half == 0)
          args.e_member[(size_t)tl.mem * args.rows_cap + my_row] =
              row_valid ? e_part[warp * 32 + lane] + e_part[(warp + 4) * 32 + lane] + sp.b4[tl.mem] : 0.f;
        asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");
      }
      } else {
        mbar_wait(&tfull[acc], acc_phase);  // nothing to drain, but the accumulator hand-shake goes on
        tc_fence_after();
      }
      // hand the accumulator back: one elected arrival per warp (on the leader's barrier in a pair)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR && rank != 0)
          mbar_arrive_remote(&tempty[acc], 0);
        else
          mbar_arrive(&tempty[acc]);
      }
      if (threadIdx.x == 0) stamp(tloc, 2, 2);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (ANI_OPND_FP16X2 && args.status && !(omax <= OPND_HALF_MAX)) atomicOr(args.status, ANI_STATUS_OPERAND_RANGE);
  }

  // ---- teardown
  if (warp < NUM_EPI_WARPS && lane == 0) bulk_wait_all();  // outstanding TMA stores are complete
  tc_fence_before();
  if (PAIR)
    cluster_sync_all();  // neither CTA leaves (or frees tensor memory) while the other still works
  else
    __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    if (PAIR)
      tmem_dealloc2(tmem_base, TMEM_COLS);
    else
      tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc
}  // namespace ani
