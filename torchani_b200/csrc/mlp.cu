// Ensemble MLP forward + backward-to-input on the species-grouped AEV matrix.
//
// Replaces nn/_containers.py:377-421,608-651 (per-species gather / 8-member python loop),
// nn/_infer.py:61-216 (BmmEnsemble) and csrc/mnp.cpp:63-236 (mnp::run).  The rows of the AEV
// matrix are already grouped by species in 128-row tiles (ani_b200_species_layout), so every
// layer of every member of every species is one grouped GEMM launch:
//     C[tile rows, N] = epilogue(A[tile rows, K] x B[K, N])
// The 8 ensemble members share the layer-1 input, so layer 1 is one GEMM with the members
// concatenated along N (the AEV is read once, not 8x as in BmmLinear's expand()).
// Backward-to-input runs the same kernel on the transposed weights; CELU'(x) is recovered
// from the stored activation y as (y > 0 ? 1 : (y + alpha) / alpha)  (csrc/mnp.cpp:206-209).
//
// Arithmetic: tcgen05 tensor cores on fp32-accurate 16-bit operand pieces (2 x fp16 with power-of-two
// operand scales, or 3 x bf16; gemm_tc.cuh / common.cuh).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gemm_tc.cuh"
#include "gemm_fused.cuh"
#include "gemm_chain.cuh"
#include "gemm_resident.cuh"

namespace ani {

// per-conformer reduction of atomic energies (fp64 accumulation) + self energies (sae.py:54-64)
struct ReduceArgs {
  const float* e_member;
  int rows_cap;
  const int32_t* row_of;
  const int32_t* orig_to_sorted;
  const int32_t* species;
  int n, lo, hi, n_per_conf;
  const double* sae;
  float* atomic_out;
  float* member_atomic_out;
  double* energies_out;
  int num_members;
  float member_scale[ANI_MAX_MEMBERS];
};

__global__ void __launch_bounds__(256) k_reduce_energies(const __grid_constant__ ReduceArgs args) {
  // one thread per atom; conformer sums by warp-aggregated float64 atomics (energies_out is
  // zeroed by the launcher)
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in_range = a < args.n;
  double contrib = 0.0;
  int conf = -1;
  if (in_range) {
    conf = a / args.n_per_conf;
    const int sp = args.species[a];
    float e = 0.f;
    bool owned = false;
    int row = 0;
    if (sp >= 0) {
      const int i = args.orig_to_sorted[a];
      if (i >= args.lo && i < args.hi) {
        owned = true;
        row = args.row_of[i];
      }
    }
    for (int m = 0; m < args.num_members; ++m) {
      const float em = owned ? args.e_member[(size_t)m * args.rows_cap + row] : 0.f;
      if (args.member_atomic_out) args.member_atomic_out[(size_t)m * args.n + a] = em;
      e += args.member_scale[m] * em;
    }
    if (args.atomic_out) args.atomic_out[a] = e;
    if (owned) contrib = (double)e + (args.sae ? args.sae[sp] : 0.0);
  }
  const int conf0 = __shfl_sync(ANI_FULL_MASK, conf, 0);
  const bool uniform = __all_sync(ANI_FULL_MASK, conf == conf0 || !in_range);
  if (uniform) {
    for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(ANI_FULL_MASK, contrib, o);
    if ((threadIdx.x & 31) == 0 && conf0 >= 0 && contrib != 0.0) atomicAdd(&args.energies_out[conf0], contrib);
  } else if (in_range && contrib != 0.0) {
    atomicAdd(&args.energies_out[conf], contrib);
  }
}

// Per step, before the backward GEMMs:
//  (a) zero the live 32-column blocks of the plain gradient matrix (the split-K layer-1 backward accumulates into it;
//      dead blocks are never read by the AEV backward kernel);
//  (b) gather the live column blocks of the layer-1 backward operand B = W1^T [ldx][M*h1] of every species that has
//      rows into ani_mlp_model::b1_compact, packed exactly like a dense operand of (live blocks * 32) rows: the
//      producer warp of the GEMM then moves one K-block of B with ONE bulk copy instead of one 2 KB copy per live
//      block and piece (water: 10 per K-block, H C N O S: 40), which had made the layer-1 backward the one phase whose
//      main loop was bound by the copy-issue rate.  2.6 MB per step for water; no state carried between steps.
struct CompactArgs {
  const unsigned char* src[ANI_MAX_SPECIES];
  unsigned char* dst[ANI_MAX_SPECIES];   // nullptr: nothing to gather for this species
  int nkb[ANI_MAX_SPECIES];              // K-blocks of the operand (M * h1 / 32)
};

__global__ void __launch_bounds__(256) k_zero_live_blocks(float* dx, int ldx, const int32_t* layout_info, int num_species,
                                                          const int32_t* blocks, const __grid_constant__ CompactArgs ca) {
  const int count = blocks ? blocks[0] : ldx / 32;  // no list: every block is live
  if (dx) {
    const int rows = layout_info[4 + num_species] * ANI_TILE_ROWS;
    const long long total = (long long)rows * count * 8;  // float4 stores
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const int q = (int)(i & 7);
      const long long rb = i >> 3;
      const int b = (int)(rb % count);
      const long long row = rb / count;
      *reinterpret_cast<float4*>(dx + row * ldx + (blocks ? blocks[1 + b] : b) * 32 + q * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if (!blocks) return;
  // (b) one warp per 2 KB chunk = (live block q, K-block kb, piece): 32 rows x 64 B, contiguous on both sides
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n_c = count * 32;
  for (int s = 0; s < num_species; ++s) {
    if (!ca.dst[s] || layout_info[4 + s + 1] <= layout_info[4 + s]) continue;
    const int nkb = ca.nkb[s], per_q = nkb * OPND_PARTS;
    for (int c = gwarp; c < count * per_q; c += nwarps) {
      const int q = c / per_q, rem = c - q * per_q, kb = rem / OPND_PARTS, pc = rem - kb * OPND_PARTS;
      const int row0 = blocks[1 + q] * 32, n0s = row0 / tc::TN_MAX * tc::TN_MAX, bns = min(tc::TN_MAX, ldx - n0s);
      const int cr0 = q * 32, n0c = cr0 / tc::TN_MAX * tc::TN_MAX, bnc = min(tc::TN_MAX, n_c - n0c);
      const unsigned char* src = ca.src[s] + ((size_t)n0s * nkb + (size_t)kb * bns) * (OPND_PARTS * OPND_ROW_BYTES) +
                                 (size_t)pc * bns * OPND_ROW_BYTES + (size_t)(row0 - n0s) * OPND_ROW_BYTES;
      unsigned char* dst = ca.dst[s] + ((size_t)n0c * nkb + (size_t)kb * bnc) * (OPND_PARTS * OPND_ROW_BYTES) +
                           (size_t)pc * bnc * OPND_ROW_BYTES + (size_t)(cr0 - n0c) * OPND_ROW_BYTES;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        reinterpret_cast<uint4*>(dst)[j * 32 + lane] = __ldg(reinterpret_cast<const uint4*>(src) + j * 32 + lane);
    }
  }
}


// ---- model-pack time: plain fp32 weights -> tiled B operand (include/ani_b200.h section 6) ----
// One thread per (output row n, 8-column chunk of K): splits scale * W into the 16-bit pieces and stores one
// 16-byte chunk per piece at its swizzled place.  `transpose`: B[n][k] = src[k][n] (the backward operands are the
// transposed weights); K is zero-padded to a multiple of 32; blockIdx.z = ensemble member (batched operands).
__global__ void __launch_bounds__(256) k_pack_b_operand(const float* __restrict__ src, int N, int K, int ld_src,
                                                        int transpose, float scale, long long src_batch_stride,
                                                        unsigned char* __restrict__ dst, long long dst_batch_stride) {
  const int kp = (K + 31) / 32 * 32, nkb = kp / 32, chunks = kp / 8;
  const long long total = (long long)N * chunks;
  const float* s = src + (long long)blockIdx.z * src_batch_stride;
  unsigned char* d = dst + (long long)blockIdx.z * dst_batch_stride;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(t / chunks), c8 = (int)(t % chunks);
    const int n0 = n / 256 * 256, bn = min(256, N - n0), r = n - n0;
    const int kb = c8 >> 2, ch = c8 & 3;
    uint32_t w[4][OPND_PARTS];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int k = c8 * 8 + 2 * i + j;
        v[j] = k < K ? scale * (transpose ? s[(long long)k * ld_src + n] : s[(long long)n * ld_src + k]) : 0.f;
      }
      tc::split_pair(v[0], v[1], w[i]);
    }
    unsigned char* blk = d + ((size_t)n0 * nkb + (size_t)kb * bn) * (OPND_PARTS * OPND_ROW_BYTES);
    const uint32_t off = (uint32_t)(r >> 3) * 512u + (uint32_t)(r & 7) * 64u + (uint32_t)((ch ^ ((r >> 1) & 3)) << 4);
#pragma unroll
    for (int p = 0; p < OPND_PARTS; ++p)
      *reinterpret_cast<uint4*>(blk + (size_t)p * bn * OPND_ROW_BYTES + off) = make_uint4(w[0][p], w[1][p], w[2][p], w[3][p]);
  }
}

}  // namespace ani

using namespace ani;

// timing experiments: clock64 stamps of the first CTAs of the next GEMM launches
static long long* g_trace = nullptr;
static int g_trace_launches = 0, g_trace_next = 0;
constexpr int TRACE_WORDS_PER_LAUNCH = 4 * 8 * 3 * 4;

extern "C" int ani_b200_debug_gemm_trace(long long* buf, int launches) {
  g_trace = buf;
  g_trace_launches = buf ? launches : 0;
  g_trace_next = 0;
  return ANI_OK;
}

// tensor-core launch: one persistent CTA per SM walks the device-side tile list
// `dependent`: launch with programmatic stream serialisation (PDL) -- the CTAs of this launch may be
// scheduled while the previous kernel of the stream drains (its CTAs occupy a whole SM each, so a
// new CTA starts as soon as one of them exits), run their prologue (barriers, tensor memory, tile
// map) and block in griddepcontrol.wait until the previous grid has completed and flushed.
template <int EPI>
static void launch_gemm_tc(const tc::Args& a_in, cudaStream_t st, bool dependent = false, bool allow_pair = true) {
  tc::Args a = a_in;
  a.trace = nullptr;
  if (g_trace && g_trace_next < g_trace_launches) a.trace = g_trace + (size_t)(g_trace_next++) * TRACE_WORDS_PER_LAUNCH;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  static const bool pdl = []() {
    const char* e = getenv("ANI_B200_PDL");  // ANI_B200_PDL=0: plain stream order
    return !e || atoi(e) != 0;
  }();
  // CTA pairs (cta_group::2, clusters of 2): each SM loads half of B.  ANI_B200_GEMM_PAIR=1 switches
  // it on for the dense launches (the block-sparse layer-1 backward gathers B in 32-row blocks and
  // stays single)
  static const bool pair_env = []() {
    const char* e = getenv("ANI_B200_GEMM_PAIR");
    return e && atoi(e) != 0;
  }();
  const bool pair = pair_env && allow_pair && EPI != tc::EPI_PLAIN && a.nblocks == nullptr;
  auto k1 = tc::k_gemm_tc<EPI, false>;
  auto k2 = tc::k_gemm_tc<(EPI == tc::EPI_PLAIN ? tc::EPI_BIAS_CELU : EPI), true>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES);
    cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES);
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pair ? (num_sms & ~1) : num_sms);
  cfg.blockDim = dim3(tc::THREADS);
  cfg.dynamicSmemBytes = tc::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (dependent && pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (pair) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  if (pair)
    cudaLaunchKernelEx(&cfg, k2, a);
  else
    cudaLaunchKernelEx(&cfg, k1, a);
}

extern "C" int ani_b200_pack_b_operand(const float* src, int n, int k, int ld_src, int transpose, float scale,
                                       int batch, long long src_batch_stride, void* dst, long long dst_batch_stride,
                                       void* stream) {
  if (!src || !dst || n < 32 || n % 32 || k < 1 || batch < 1 || !(scale > 0.f)) return ANI_ERR_BAD_ARG;
  const long long total = (long long)n * ((k + 31) / 32 * 4);
  const int blocks = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
  k_pack_b_operand<<<dim3(blocks, 1, batch), 256, 0, (cudaStream_t)stream>>>(src, n, k, ld_src, transpose, scale,
                                                                              src_batch_stride,
                                                                              static_cast<unsigned char*>(dst),
                                                                              dst_batch_stride);
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}

// shared argument checks + the launch-invariant part of the GEMM arguments
static int mlp_common(const ani_mlp_model* model, int rows_cap, const int32_t* row_atom, const int32_t* layout_info,
                      void* act1, void* act2, void* act3, int32_t* status, tc::Args& ta) {
  if (!model || !row_atom || !layout_info || !act1 || !act2 || !act3) return ANI_ERR_BAD_ARG;
  const int S = model->num_species, M = model->num_members;
  if (S < 1 || S > ANI_MAX_SPECIES || M < 1 || M > ANI_MAX_MEMBERS) return ANI_ERR_BAD_ARG;
  if (rows_cap < ANI_TILE_ROWS || rows_cap % ANI_TILE_ROWS) return ANI_ERR_BAD_ARG;
  const int ldx = model->ldx;
  if (ldx % 32 || ldx < model->in_dim) return ANI_ERR_BAD_ARG;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    if (p.h1 % 32 || p.h2 % 32 || p.h3 % 32 || p.h1 < 32 || p.h2 < 32 || p.h3 < 32) return ANI_ERR_UNSUPPORTED;
    if (p.h1 > model->h1_max || p.h2 > model->h2_max || p.h3 > model->h3_max) return ANI_ERR_BAD_ARG;
    if (p.h3 > tc::TN_MAX) return ANI_ERR_UNSUPPORTED;  // the fused final layer needs h3 in one accumulator
    if (!p.b1 || !p.b2 || !p.b3 || !p.w4 || !p.b4 || !p.t_f1 || !p.t_f2 || !p.t_f3 || !p.t_b3 || !p.t_b2 || !p.t_b1)
      return ANI_ERR_BAD_ARG;
    for (int l = 0; l < 3; ++l)
      if (ANI_OPND_FP16X2 && !(p.w_scale[l] > 0.f)) return ANI_ERR_BAD_ARG;
  }
  ta.layout_info = layout_info;
  ta.kblocks = nullptr;
  ta.nblocks = nullptr;
  ta.num_species = S;
  ta.alpha = model->celu_alpha;
  ta.e_member = nullptr;
  ta.row_atom = row_atom;
  ta.rows_cap = rows_cap;
  ta.want_backward = 0;
  ta.ldc = 0;
  ta.c_accumulate = 0;
  static const int gemm_debug = []() {
    const char* e = getenv("ANI_B200_GEMM_DEBUG");  // timing experiments only: results are wrong when set
    return e ? atoi(e) : 0;
  }();
  ta.debug = gemm_debug;
  for (int m = 0; m < ANI_MAX_MEMBERS; ++m) ta.member_scale[m] = m < M ? model->member_scale[m] : 0.f;
  for (int s = 0; s < ANI_MAX_SPECIES; ++s) ta.sp[s] = tc::Species{nullptr, nullptr, 0, 0, 0, 0, 0, nullptr, nullptr, 0, 0, 1.0f};
  ta.status = status;
  static const int narrow = []() {
    const char* e = getenv("ANI_B200_NARROW_TILES");  // 0: 256-column tiles whatever the list length
    return !e || atoi(e) != 0;
  }();
  ta.allow_narrow = narrow;
  ta.b_compact = 0;
  ta.win_idx = 0;
  ta.win_cnt = 1;
  static const int epi_direct = []() {
    const char* e = getenv("ANI_B200_EPI_DIRECT");  // 0: shared-memory staging + TMA bulk stores (round 1 / early round 2)
    return !e || atoi(e) != 0;
  }();
  ta.epi_direct = epi_direct;
  ta.out_scale = OPND_SCALE_VALUE;
  ta.y_inv_scale = 1.0f / OPND_SCALE_VALUE;
  return ANI_OK;
}

// Layer-1 backward dX = sum_m G1_m x W1_m: how many members one work unit contracts in its own accumulator (the
// rest of the sum goes through vector REDs into dx).  1 = round 1 (one unit per member: most parallelism, 8 partial
// sums per element); larger groups halve / quarter the RED traffic and the per-unit ramp at the price of fewer units.
// Measured on B200 (profiles/r02_sweep.md, run 16; step ms at G = 1 / 2 / 4): 999 atoms 0.147 / 0.150 / 0.158,
// 9 999 atoms 0.373 / 0.364 / 0.367, 49 999 atoms 2.062 / 1.960 / 1.929 -> by row capacity unless the env pins it.
static int l1b_group(int M, int rows_cap) {
  static const int env = []() {
    const char* e = getenv("ANI_B200_L1B_GROUP");
    return e ? atoi(e) : 0;
  }();
  int g = env >= 1 ? env : (rows_cap < 4096 ? 1 : rows_cap < 32768 ? 2 : 4);
  while (g > 1 && M % g) --g;
  return g;
}

// operand scales (common.cuh): activations / AEVs carry sv, gradients sg, weights their per-tensor
// w_scale; every GEMM divides the product of its two operand scales out of the accumulator
static inline float wsc(const ani_mlp_species& p, int layer) { return ANI_OPND_FP16X2 ? p.w_scale[layer] : 1.0f; }

// compacted layer-1 backward operands (k_zero_live_blocks (b)): species s starts where the full operands of the species
// before it would end -- ani_mlp_model::b1_compact holds sum_s ldx * (M h1_s / 32) * P * 64 bytes
static bool use_b1_compact(const ani_mlp_model* model, const int32_t* aev_blocks) {
  static const bool on = []() {
    const char* e = getenv("ANI_B200_B1_COMPACT");  // 0: gather the live blocks with 2 KB copies inside the GEMM
    return !e || atoi(e) != 0;
  }();
  return on && model->b1_compact && aev_blocks;
}
static unsigned char* b1_compact_ptr(const ani_mlp_model* model, int s) {
  size_t off = 0;
  for (int t = 0; t < s; ++t)
    off += (size_t)model->ldx * (size_t)(model->num_members * model->sp[t].h1 / 32) * (OPND_PARTS * OPND_ROW_BYTES);
  return static_cast<unsigned char*>(model->b1_compact) + off;
}
// zero-fill of dE/dAEV (dx may be NULL: nothing to zero) + gather of the compact operands
static void launch_zero_compact(const ani_mlp_model* model, float* dx, const int32_t* layout_info, const int32_t* aev_blocks,
                                cudaStream_t st) {
  CompactArgs ca;
  const bool compact = use_b1_compact(model, aev_blocks);
  for (int s = 0; s < ANI_MAX_SPECIES; ++s) {
    const bool live = compact && s < model->num_species;
    ca.src[s] = live ? static_cast<const unsigned char*>(model->sp[s].t_b1) : nullptr;
    ca.dst[s] = live ? b1_compact_ptr(model, s) : nullptr;
    ca.nkb[s] = live ? model->num_members * model->sp[s].h1 / 32 : 0;
  }
  if (!dx && !compact) return;
  k_zero_live_blocks<<<592, 256, 0, st>>>(dx, model->ldx, layout_info, model->num_species, aev_blocks, ca);
}

extern "C" int ani_b200_mlp_forward(const ani_mlp_model* model, const void* x, int rows_cap, const int32_t* row_atom,
                                    const int32_t* layout_info, const int32_t* aev_blocks, void* act1, void* act2,
                                    void* act3, float* e_member, int want_backward, int32_t* status, void* stream) {
  if (!x || !e_member) return ANI_ERR_BAD_ARG;
  tc::Args ta;
  const int rc = mlp_common(model, rows_cap, row_atom, layout_info, act1, act2, act3, status, ta);
  if (rc != ANI_OK) return rc;
  const int S = model->num_species, M = model->num_members, ldx = model->ldx;
  const float sv = OPND_SCALE_VALUE, sg = OPND_SCALE_GRAD;
  cudaStream_t st = (cudaStream_t)stream;
  // 32-column blocks per row of the tiled activation matrices
  const int kb1 = M * model->h1_max / 32, kb2 = M * model->h2_max / 32, kb3 = M * model->h3_max / 32, kbx = ldx / 32;
  ta.e_member = e_member;
  ta.want_backward = want_backward;
  // Layer 1: the members share the input (A offset 0 for every member), one GEMM per member like the other layers
  ta.A = static_cast<const unsigned char*>(x); ta.a_kblocks = kbx; ta.C = act1; ta.c_kblocks = kb1; ta.members = M;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f1), p.b1, ldx, p.h1, 0, p.h1, p.h1, nullptr, nullptr, 0, 0,
                            1.0f / (sv * wsc(p, 0))};
  }
  ta.kblocks = aev_blocks;  // dead AEV column blocks contribute exact zeros: skip them
  launch_gemm_tc<tc::EPI_BIAS_CELU>(ta, st);
  ta.kblocks = nullptr;
  ta.A = static_cast<const unsigned char*>(act1); ta.a_kblocks = kb1; ta.C = act2; ta.c_kblocks = kb2; ta.members = M;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f2), p.b2, p.h1, p.h2, p.h1, p.h2, p.h2, nullptr, nullptr, 0, 0,
                            1.0f / (sv * wsc(p, 1))};
  }
  launch_gemm_tc<tc::EPI_BIAS_CELU>(ta, st, true);
  ta.A = static_cast<const unsigned char*>(act2); ta.a_kblocks = kb2; ta.C = act3; ta.c_kblocks = kb3; ta.members = M;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f3), p.b3, p.h2, p.h3, p.h2, p.h3, p.h3, p.w4, p.b4, 0, 0,
                            1.0f / (sv * wsc(p, 2))};
  }
  // layer 3 + final layer (h3 -> 1) + gradient seed, fused in the epilogue: act3 receives
  // G3 = scale_m * w4 * celu'(a3) directly, e_member the per-member atomic energies
  ta.out_scale = sg;  // act3 receives the gradient seed
  ta.allow_narrow = 0;  // the fused final layer needs all of h3 in one accumulator
  launch_gemm_tc<tc::EPI_HEAD>(ta, st, true);
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}

extern "C" int ani_b200_zero_live_blocks(const ani_mlp_model* model, float* dx, const int32_t* layout_info,
                                         const int32_t* aev_blocks, void* stream) {
  if (!model || !dx || !layout_info) return ANI_ERR_BAD_ARG;
  launch_zero_compact(model, dx, layout_info, aev_blocks, (cudaStream_t)stream);
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}

extern "C" int ani_b200_mlp_backward(const ani_mlp_model* model, float* dx, int rows_cap, const int32_t* row_atom,
                                     const int32_t* layout_info, const int32_t* aev_blocks, void* act1, void* act2,
                                     void* act3, int dx_zeroed, int32_t* status, void* stream) {
  if (!dx) return ANI_ERR_BAD_ARG;
  tc::Args ta;
  const int rc = mlp_common(model, rows_cap, row_atom, layout_info, act1, act2, act3, status, ta);
  if (rc != ANI_OK) return rc;
  const int S = model->num_species, M = model->num_members, ldx = model->ldx;
  const float sg = OPND_SCALE_GRAD;
  cudaStream_t st = (cudaStream_t)stream;
  const int kb1 = M * model->h1_max / 32, kb2 = M * model->h2_max / 32, kb3 = M * model->h3_max / 32;
  ta.want_backward = 1;
  ta.out_scale = sg;
  // G2 = (G3 x W3) * celu'(A2), G1 = (G2 x W2) * celu'(A1), dX = G1 x W1
  ta.A = static_cast<const unsigned char*>(act3); ta.a_kblocks = kb3; ta.C = act2; ta.c_kblocks = kb2; ta.members = M;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b3), nullptr, p.h3, p.h2, p.h3, p.h2, 0, nullptr, nullptr, 0, 0,
                            1.0f / (sg * wsc(p, 2))};
  }
  // (after a cross-stream join -- the caller zeroed dx elsewhere -- the first launch is a plain one)
  launch_gemm_tc<tc::EPI_MUL_DCELU>(ta, st, !dx_zeroed);
  ta.A = static_cast<const unsigned char*>(act2); ta.a_kblocks = kb2; ta.C = act1; ta.c_kblocks = kb1; ta.members = M;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b2), nullptr, p.h2, p.h1, p.h2, p.h1, 0, nullptr, nullptr, 0, 0,
                            1.0f / (sg * wsc(p, 1))};
  }
  launch_gemm_tc<tc::EPI_MUL_DCELU>(ta, st, true);
  // dX = sum_m G1_m x W1_m: split-K over the members (one work unit per (row tile, member), so
  // all SMs are busy even when there are fewer row tiles than SMs); the partial tiles are
  // accumulated with vector REDs into the zeroed live column blocks of dx
  const int G = l1b_group(M, rows_cap);
  ta.A = static_cast<const unsigned char*>(act1); ta.a_kblocks = kb1; ta.C = dx; ta.c_kblocks = 0; ta.ldc = ldx; ta.members = M / G;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b1), nullptr, G * p.h1, ldx, G * p.h1, 0, 0, nullptr, nullptr,
                            M * p.h1 / 32, G * p.h1 / 32, 1.0f / (sg * wsc(p, 0))};
  }
  ta.nblocks = aev_blocks;  // ... and nobody reads the gradient of a dead column block
  ta.c_accumulate = M / G > 1;
  if (use_b1_compact(model, aev_blocks)) {
    ta.b_compact = 1;
    for (int s = 0; s < S; ++s) ta.sp[s].Bt = b1_compact_ptr(model, s);
  }
  // (ani_b200_zero_live_blocks, if the caller ran it for this step, has also gathered the compact operands)
  if (!dx_zeroed) launch_zero_compact(model, ta.c_accumulate ? dx : nullptr, layout_info, aev_blocks, st);
  launch_gemm_tc<tc::EPI_PLAIN>(ta, st, true);
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}

// ---- the whole MLP of a step as ONE persistent data-flow launch (gemm_fused.cuh) ----------------------
// phase p of the list: 0-2 forward layers (2 = head), 3-5 backward-to-input.  `sync`: 6 * (rows_cap / 128) ints.
static void fill_phase(tc::Args& ta, int phase, const ani_mlp_model* model, const void* x, float* dx, void* act1,
                       void* act2, void* act3, float* e_member, const int32_t* aev_blocks, int want_backward,
                       int rows_cap = 0, int group_override = 0) {
  const int S = model->num_species, M = model->num_members, ldx = model->ldx;
  const float sv = OPND_SCALE_VALUE, sg = OPND_SCALE_GRAD;
  const int kb1 = M * model->h1_max / 32, kb2 = M * model->h2_max / 32, kb3 = M * model->h3_max / 32, kbx = ldx / 32;
  ta.kblocks = nullptr;
  ta.nblocks = nullptr;
  ta.e_member = e_member;
  ta.want_backward = want_backward;
  ta.c_accumulate = 0;
  ta.ldc = 0;
  ta.out_scale = sv;
  ta.y_inv_scale = 1.0f / sv;
  for (int s = 0; s < S; ++s) {
    const ani_mlp_species& p = model->sp[s];
    switch (phase) {
      case 0:
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f1), p.b1, ldx, p.h1, 0, p.h1, p.h1, nullptr, nullptr, 0, 0,
                                1.0f / (sv * wsc(p, 0))};
        break;
      case 1:
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f2), p.b2, p.h1, p.h2, p.h1, p.h2, p.h2, nullptr, nullptr, 0, 0,
                                1.0f / (sv * wsc(p, 1))};
        break;
      case 2:
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_f3), p.b3, p.h2, p.h3, p.h2, p.h3, p.h3, p.w4, p.b4, 0, 0,
                                1.0f / (sv * wsc(p, 2))};
        break;
      case 3:
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b3), nullptr, p.h3, p.h2, p.h3, p.h2, 0, nullptr, nullptr, 0, 0,
                                1.0f / (sg * wsc(p, 2))};
        break;
      case 4:
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b2), nullptr, p.h2, p.h1, p.h2, p.h1, 0, nullptr, nullptr, 0, 0,
                                1.0f / (sg * wsc(p, 1))};
        break;
      default: {
        const int G = (want_backward == 2 || group_override) ? max(1, group_override) : l1b_group(M, rows_cap);
        ta.sp[s] = tc::Species{static_cast<const unsigned char*>(p.t_b1), nullptr, G * p.h1, ldx, G * p.h1, 0, 0, nullptr, nullptr,
                                M * p.h1 / 32, G * p.h1 / 32, 1.0f / (sg * wsc(p, 0))};
        break;
      }
    }
  }
  switch (phase) {
    case 0: ta.A = static_cast<const unsigned char*>(x); ta.a_kblocks = kbx; ta.C = act1; ta.c_kblocks = kb1; ta.members = M;
            ta.kblocks = aev_blocks; break;
    case 1: ta.A = static_cast<const unsigned char*>(act1); ta.a_kblocks = kb1; ta.C = act2; ta.c_kblocks = kb2; ta.members = M; break;
    case 2: ta.A = static_cast<const unsigned char*>(act2); ta.a_kblocks = kb2; ta.C = act3; ta.c_kblocks = kb3; ta.members = M;
            ta.out_scale = sg; ta.allow_narrow = 0; break;
    case 3: ta.A = static_cast<const unsigned char*>(act3); ta.a_kblocks = kb3; ta.C = act2; ta.c_kblocks = kb2; ta.members = M;
            ta.out_scale = sg; break;
    case 4: ta.A = static_cast<const unsigned char*>(act2); ta.a_kblocks = kb2; ta.C = act1; ta.c_kblocks = kb1; ta.members = M;
            ta.out_scale = sg; break;
    default: ta.A = static_cast<const unsigned char*>(act1); ta.a_kblocks = kb1; ta.C = dx; ta.c_kblocks = 0; ta.ldc = ldx;
            ta.members = M / ((want_backward == 2 || group_override) ? max(1, group_override) : l1b_group(M, rows_cap));
            ta.nblocks = aev_blocks;
            ta.c_accumulate = ta.members > 1; ta.out_scale = sg; break;
  }
  if (phase == 5 && use_b1_compact(model, aev_blocks)) {
    ta.b_compact = 1;
    for (int s = 0; s < S; ++s) ta.sp[s].Bt = b1_compact_ptr(model, s);
  }
  if (phase == 5 && want_backward == 2) {
    // per-member dE_m/dAEV: member m writes its own [rows_cap][ldx] slab of dx (plain stores, no accumulation)
    ta.c_accumulate = 0;
    for (int s = 0; s < S; ++s) ta.sp[s].c_moff = rows_cap * ldx;
  }
}

// number of row-tile windows (= launches of the data-flow kernel) ani_b200_mlp_step cuts a step into
static bool use_chain_launch(const ani_mlp_model* model) {
  // Opt-in (ANI_B200_MLP_CHAIN=1).  Measured on B200 (profiles/r02_sweep.md): 224 us at 9 999 atoms whatever the
  // interleave depth against 215 us for the phase-major launch, 94 vs 76 us (chained launches) at 999 atoms, 1.41 vs
  // 1.10 ms at 50 k atoms -- all three schedules are bound by the same eight epilogue warps, and the chains give up
  // the per-phase ring geometry and the member grouping of the layer-1 backward.
  const char* ce = getenv("ANI_B200_MLP_CHAIN");
  bool ok = ce && atoi(ce) != 0;
  for (int s = 0; s < model->num_species; ++s)
    ok = ok && model->sp[s].h1 <= tc::TN_MAX && model->sp[s].h2 <= tc::TN_MAX && model->sp[s].h3 <= tc::TN_MAX;
  return ok;
}

// Shared-memory plan of the resident-chain launch (gemm_resident.cuh): the 128-row image of the widest hidden layer
// (2 x fp16: 16 KB per 32 columns; ANI-2x 256 -> 128 KB, ANI-1x 160 -> 80 KB) plus a ring of B-only stages behind it,
// at least two of a 256-column tile (32 KB; ANI-2x: 2, ANI-1x: 4 -- narrower layers get more, sized on the device); the
// layer-1 forward uses a ring of A + B stages over all of it.  Two ring stages are the least that keeps the copies
// ahead of the MMAs; 3 x bf16 operands (24 KB per K-block, 48 KB per stage) do not fit
// that and keep the other launches.
struct ResidentPlan {
  bool fits;
  int res_kb, res_bytes, small_stages, ring_bytes, big_stages;
};
static ResidentPlan resident_plan(const ani_mlp_model* model) {
  ResidentPlan pl = {false, 0, 0, 0, 0, 0};
  int hmax = 0;
  bool widths_ok = true;
  for (int s = 0; s < model->num_species; ++s) {
    const ani_mlp_species& p = model->sp[s];
    hmax = max(hmax, max(p.h1, max(p.h2, p.h3)));
    widths_ok = widths_ok && p.h1 <= tc::TN_MAX && p.h2 <= tc::TN_MAX && p.h3 <= tc::TN_MAX;
  }
  pl.res_kb = (hmax + tc::TK - 1) / tc::TK;
  pl.res_bytes = pl.res_kb * tc::A_BLOCK_BYTES;
  pl.small_stages = min(tc::MAX_STAGES, max(0, tc::RES_AVAIL - pl.res_bytes) / tc::RES_B_STAGE_BYTES);
  pl.ring_bytes = pl.small_stages * tc::RES_B_STAGE_BYTES;
  pl.big_stages = min(tc::MAX_STAGES, tc::RES_AVAIL / tc::CHAIN_STAGE_BYTES);
  pl.fits = widths_ok && hmax > 0 && pl.small_stages >= 2 && pl.big_stages >= 2;
  return pl;
}

// Where the plan fits (the opt-in ANI_B200_MLP_CHAIN=1 comes first), for lists of at most 8 chains per SM;
// ANI_B200_MLP_RESIDENT=0 / 1: never / whatever the length.  Measured on B200 (1000 W, profiles/r03_bench_*), MLP
// stage against the data-flow launch / chained launches: water 999 atoms (0.5 chains per SM) 58 vs 82 us, gdb256 121
// vs 144 us, water 9 999 atoms (4.3 per SM) 185 vs 202 us; protein in water 50 k atoms (21 per SM) 1.20 vs 1.12 ms.
static bool use_resident_launch(const ani_mlp_model* model, int rows_cap) {
  if (use_chain_launch(model) || !resident_plan(model).fits) return false;
  const char* e = getenv("ANI_B200_MLP_RESIDENT");
  if (e) return atoi(e) != 0;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      num_sms = 148;   // (host-only callers: a B200)
  }
  return (long long)(rows_cap / ANI_TILE_ROWS) * model->num_members <= 8LL * num_sms;
}

extern "C" int ani_b200_mlp_resident_plan(const ani_mlp_model* model, int32_t* out) {
  if (!model || !out || model->num_species < 1 || model->num_species > ANI_MAX_SPECIES) return ANI_ERR_BAD_ARG;
  const ResidentPlan pl = resident_plan(model);
  out[0] = pl.res_bytes;
  out[1] = pl.ring_bytes;
  out[2] = pl.big_stages * tc::CHAIN_STAGE_BYTES;
  out[3] = tc::RES_AVAIL;
  out[4] = pl.fits ? 1 : 0;
  return ANI_OK;
}

extern "C" int ani_b200_mlp_step_kernel(const ani_mlp_model* model, int rows_cap) {
  if (!model) return ANI_ERR_BAD_ARG;
  return use_chain_launch(model) ? 1 : use_resident_launch(model, rows_cap) ? 2 : 0;
}

extern "C" int ani_b200_mlp_step_windows(const ani_mlp_model* model, int rows_cap) {
  if (!model || rows_cap < ANI_TILE_ROWS) return 1;
  if (use_chain_launch(model) || use_resident_launch(model, rows_cap)) return 1;   // independent chains: one launch
  // Experiment (measured on B200, 9 999 atoms: 214 / 305 / 387 / 479 us for 1 / 2 / 3 / 4 windows): every launch of the
  // phase-major kernel costs ~90 us of dependency ramp before its ~4.9 us per unit and CTA, far more than the L2
  // residency of a window buys -- one window unless the environment asks for more
  const char* e = getenv("ANI_B200_MLP_CHUNKS");
  int chunks = e ? atoi(e) : 1;
  if (chunks < 1) chunks = 1;
  const int n_tiles_cap = rows_cap / ANI_TILE_ROWS;
  if (chunks > n_tiles_cap / 8) chunks = n_tiles_cap / 8 > 1 ? n_tiles_cap / 8 : 1;   // a window keeps >= 8 row tiles
  return chunks;
}

static int epi_warps_env() {
  static const int v = []() {
    const char* e = getenv("ANI_B200_EPI_WARPS");  // 8 (default) or 16: epilogue warps of the fused kernel
    return e && atoi(e) == 16 ? 16 : 8;
  }();
  return v;
}

extern "C" int ani_b200_mlp_step(const ani_mlp_model* model, const void* x, float* dx, int rows_cap,
                                 const int32_t* row_atom, const int32_t* layout_info, const int32_t* aev_blocks,
                                 void* act1, void* act2, void* act3, float* e_member, int want_backward,
                                 int32_t* sync_i32, int32_t* status, void* stream) {
  if (!x || !e_member || !sync_i32 || (want_backward && !dx)) return ANI_ERR_BAD_ARG;
  static tc::FusedArgs F;   // ~5 KB: built in place, passed by value (__grid_constant__)
  tc::Args base;
  const int rc = mlp_common(model, rows_cap, row_atom, layout_info, act1, act2, act3, status, base);
  if (rc != ANI_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int M = model->num_members;
  static int num_sms_c = 0;
  if (num_sms_c == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms_c, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(tc::k_mlp_chain<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::FUSED_SMEM_BYTES);
  }
  // resident chains (gemm_resident.cuh): one launch, a chain's activations and gradients in shared memory
  if (use_resident_launch(model, rows_cap)) {
    static tc::ResidentArgs RA;
    static bool attr_set = false;
    if (!attr_set) {
      cudaFuncSetAttribute(tc::k_mlp_resident, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::FUSED_SMEM_BYTES);
      attr_set = true;
    }
    const ResidentPlan pl = resident_plan(model);
    RA.n_phases = want_backward ? 6 : 3;
    RA.res_kb = pl.res_kb;
    static const int epis_r[6] = {tc::EPI_BIAS_CELU, tc::EPI_BIAS_CELU, tc::EPI_HEAD, tc::EPI_MUL_DCELU, tc::EPI_MUL_DCELU,
                                  tc::EPI_PLAIN};
    for (int p = 0; p < tc::MAX_PHASES; ++p) {
      RA.epi[p] = epis_r[p];
      RA.ph[p] = base;
      fill_phase(RA.ph[p], p, model, x, dx, act1, act2, act3, e_member, aev_blocks, want_backward, rows_cap, 1);
      RA.ph[p].allow_narrow = 0;   // one column tile per member in phases 0-4 (the layer-1 backward: any number)
    }
    if (want_backward) launch_zero_compact(model, (want_backward == 1 && M > 1) ? dx : nullptr, layout_info, aev_blocks, st);
    tc::k_mlp_resident<<<num_sms_c, tc::CHAIN_THREADS, tc::FUSED_SMEM_BYTES, st>>>(RA);
    ANI_CUDA_CHECK_LAUNCH();
    return ANI_OK;
  }
  // independent chains (gemm_chain.cuh): one launch, no synchronisation between CTAs.  ANI_B200_MLP_CHAIN=0: the
  // phase-major data-flow launch below; ANI_B200_CHAIN_DEPTH: chains a CTA interleaves
  if (use_chain_launch(model)) {
    static tc::ChainArgs CA;
    CA.n_phases = want_backward ? 6 : 3;
    const char* de = getenv("ANI_B200_CHAIN_DEPTH");
    CA.depth = de ? atoi(de) : 0;   // 0: chosen on the device from the number of chains
    if (CA.depth > tc::CHAIN_MAX_D) CA.depth = tc::CHAIN_MAX_D;
    static const int epis_c[6] = {tc::EPI_BIAS_CELU, tc::EPI_BIAS_CELU, tc::EPI_HEAD, tc::EPI_MUL_DCELU, tc::EPI_MUL_DCELU,
                                  tc::EPI_PLAIN};
    for (int p = 0; p < tc::MAX_PHASES; ++p) {
      CA.epi[p] = epis_c[p];
      CA.ph[p] = base;
      fill_phase(CA.ph[p], p, model, x, dx, act1, act2, act3, e_member, aev_blocks, want_backward, rows_cap, 1);
      CA.ph[p].allow_narrow = 0;   // a chain has one column tile per member and phase (the layer-1 backward: any number)
      CA.ph[p].epi_direct = 0;
    }
    CA.trace = nullptr;
    if (g_trace && g_trace_next == 0 && (size_t)g_trace_launches * TRACE_WORDS_PER_LAUNCH >= (size_t)4 * tc::FTRACE_UNITS * 16) {
      CA.trace = g_trace;
      g_trace_next = g_trace_launches;
    }
    if (want_backward) launch_zero_compact(model, (want_backward == 1 && M > 1) ? dx : nullptr, layout_info, aev_blocks, st);
    tc::k_mlp_chain<8><<<num_sms_c, tc::CHAIN_THREADS, tc::FUSED_SMEM_BYTES, st>>>(CA);
    ANI_CUDA_CHECK_LAUNCH();
    return ANI_OK;
  }
  F.n_phases = want_backward ? 6 : 3;
  static const int epis[6] = {tc::EPI_BIAS_CELU, tc::EPI_BIAS_CELU, tc::EPI_HEAD, tc::EPI_MUL_DCELU, tc::EPI_MUL_DCELU,
                              tc::EPI_PLAIN};
  for (int p = 0; p < tc::MAX_PHASES; ++p) {
    F.epi[p] = epis[p];
    F.dep[p] = p - 1;
    F.ph[p] = base;
    fill_phase(F.ph[p], p, model, x, dx, act1, act2, act3, e_member, aev_blocks, want_backward, rows_cap);
    F.ph[p].epi_direct = 0;   // the data-flow launch keeps the staged stores (gemm_fused.cuh)
  }
  static const int prefetch_b = []() {
    const char* e = getenv("ANI_B200_PREFETCH_B");  // 1: issue a unit's weight copies before waiting for its inputs
    return e && atoi(e) != 0;                       // (measured on B200: no gain at 1k atoms, -4 % at 10k: off)
  }();
  F.prefetch_b = prefetch_b;
  {
    const char* pe = getenv("ANI_B200_EPI16_PAIRS");   // 1: the paired sixteen-warp epilogue with staged stores
    F.epi_direct16 = epi_warps_env() == 16 && !(pe && atoi(pe) != 0);
  }
  // role timeline of the first CTAs (tools/gemm_trace.py): needs the whole six-launch buffer
  F.trace = nullptr;
  if (g_trace && g_trace_next == 0 && (size_t)g_trace_launches * TRACE_WORDS_PER_LAUNCH >= (size_t)4 * tc::FTRACE_UNITS * 16) {
    F.trace = g_trace;
    g_trace_next = g_trace_launches;
  }
  F.sync = sync_i32;
  F.sync_stride = rows_cap / ANI_TILE_ROWS;
  cudaMemsetAsync(sync_i32, 0, sizeof(int32_t) * (size_t)tc::MAX_PHASES * F.sync_stride, st);
  if (want_backward) launch_zero_compact(model, (want_backward == 1 && M > 1) ? dx : nullptr, layout_info, aev_blocks, st);
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(tc::k_mlp_fused<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::FUSED_SMEM_BYTES);
    cudaFuncSetAttribute(tc::k_mlp_fused<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::FUSED_SMEM_BYTES);
  }
  const int epi_warps = epi_warps_env();
  // The activations of a step (act1..3: 19.5 KB per row for ANI-2x x 8) outgrow the 126 MB L2 beyond ~6 k atoms: the
  // layers then stream through HBM (ncu at 10 k atoms: 554 MB of DRAM traffic per launch, L2 hit rate 60 %).  The
  // launch is therefore cut into windows of the row tiles -- all six phases of one window, then the next -- sized so
  // that a window's activations stay in the L2 between the phase that writes them and the phases that read them.
  const int chunks = ani_b200_mlp_step_windows(model, rows_cap);
  for (int c = 0; c < chunks; ++c) {
    for (int p = 0; p < tc::MAX_PHASES; ++p) {
      F.ph[p].win_idx = c;
      F.ph[p].win_cnt = chunks;
    }
    if (epi_warps == 16)
      tc::k_mlp_fused<16><<<num_sms, tc::fused_threads(16), tc::FUSED_SMEM_BYTES, st>>>(F);
    else
      tc::k_mlp_fused<8><<<num_sms, tc::fused_threads(8), tc::FUSED_SMEM_BYTES, st>>>(F);
    if (F.trace) F.trace = nullptr;   // (the role timeline records the first window)
  }
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}

extern "C" int ani_b200_mlp_forward_backward(const ani_mlp_model* model, const void* x, float* dx, int rows_cap,
                                             const int32_t* row_atom, const int32_t* layout_info,
                                             const int32_t* aev_blocks, void* act1, void* act2, void* act3,
                                             float* e_member, int want_backward, int32_t* status, void* stream) {
  if (want_backward && !dx) return ANI_ERR_BAD_ARG;
  int rc = ani_b200_mlp_forward(model, x, rows_cap, row_atom, layout_info, aev_blocks, act1, act2, act3, e_member,
                                want_backward, status, stream);
  if (rc != ANI_OK || !want_backward) return rc;
  return ani_b200_mlp_backward(model, dx, rows_cap, row_atom, layout_info, aev_blocks, act1, act2, act3, 0, status,
                               stream);
}

extern "C" int ani_b200_reduce_energies(const ani_mlp_model* model, const float* e_member, int rows_cap,
                                        const int32_t* row_of, const int32_t* orig_to_sorted,
                                        const int32_t* species, int n, int lo, int hi, int n_conf, int n_per_conf,
                                        const double* sae, float* atomic_out, float* member_atomic_out,
                                        double* energies_out, void* stream) {
  if (!model || !e_member || !row_of || !orig_to_sorted || !species || !energies_out) return ANI_ERR_BAD_ARG;
  if (n != n_conf * n_per_conf || n_conf < 1) return ANI_ERR_BAD_ARG;
  ReduceArgs ra;
  ra.e_member = e_member; ra.rows_cap = rows_cap; ra.row_of = row_of; ra.orig_to_sorted = orig_to_sorted;
  ra.species = species; ra.n = n; ra.lo = lo; ra.hi = hi; ra.n_per_conf = n_per_conf; ra.sae = sae;
  ra.atomic_out = atomic_out; ra.member_atomic_out = member_atomic_out; ra.energies_out = energies_out;
  ra.num_members = model->num_members;
  for (int m = 0; m < ANI_MAX_MEMBERS; ++m)
    ra.member_scale[m] = m < model->num_members ? model->member_scale[m] : 0.f;
  cudaMemsetAsync(energies_out, 0, sizeof(double) * (size_t)n_conf, (cudaStream_t)stream);
  k_reduce_energies<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ra);
  ANI_CUDA_CHECK_LAUNCH();
  return ANI_OK;
}
