/*
 * ani_b200.h -- C-ABI of the B200-native ANI energy+force hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Every entry point takes plain device
 * pointers, sizes and an explicit cudaStream_t (passed as void*), never allocates,
 * never synchronises the host, and returns 0 on success or a negative ANI_ERR_* code
 * (ani_b200_error_string() explains it).  Device-side conditions that the reference
 * reports as exceptions (neighbour overflow, periodic cell smaller than the cutoff)
 * are raised through a device status word that the caller reads when convenient.
 *
 * What each entry point replaces in the reference (paths under /root/reference/torchani):
 *   ani_b200_build_cells        neighbors.py:418-507,554-615 (_cell_list bucketing), utils.py:237-255
 *                               (map_to_central), csrc/cell_list.cpp:266-350
 *   ani_b200_species_layout     nn/_containers.py:412-415 (per-species nonzero/index_select)
 *   ani_b200_active_aev_blocks  (no counterpart: exact block-sparsity of the AEV the reference ignores)
 *   ani_b200_aev_forward        neighbors.py:64-113,968-1002 + aev/_computer.py:274-350;
 *                               csrc/cuaev.cpp:189-246 (cuaev::run / run_with_half_nbrlist),
 *                               csrc/aev.cu:323-472,768-834 (K8/K9), :975-1039 (K4)
 *   ani_b200_aev_backward       csrc/cuaev.cpp:134-163, csrc/aev.cu:474-766,837-967 (K10/K11)
 *   ani_b200_pairs_to_rows, ani_b200_aev_*_rows   aev/_computer.py:251-272, csrc/aev.cu:1128-1208 (K6)
 *   ani_b200_half_neighbor_*    neighbors.py:366-415 (cell_list), :187-212 (all_pairs) -> Neighbors
 *   ani_b200_mlp_forward_backward  nn/_containers.py:377-421,608-651, nn/_core.py:146-167,
 *                               nn/_infer.py:61-216 (BmmEnsemble), csrc/mnp.cpp:63-236 (mnp::run)
 *   ani_b200_mlp_forward / _zero_live_blocks / _mlp_backward   the same, as separate halves
 *   ani_b200_reduce_energies    nn/_containers.py:418-421,633-636, sae.py:54-64
 *   ani_b200_verlet_positions   neighbors.py:759-884 (VerletCellList: reuse of a list built with a skin)
 *   ani_b200_aev_backward(..., virial, ...)   ase.py:164-168 (the "f dot r" virial of the stress)
 *   ani_b200_operand_format     (no counterpart: format of the tensor-core GEMM operands of this build)
 */
#ifndef ANI_B200_H
#define ANI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ANI_B200_ABI_VERSION 4

#define ANI_MAX_SPECIES 8
#define ANI_MAX_SHFR 32
#define ANI_MAX_SHFA 8
#define ANI_MAX_SHFZ 8
#define ANI_MAX_MEMBERS 16
#define ANI_TILE_ROWS 128 /* rows of the species-grouped AEV matrix per MLP tile */

/* error codes (return values) */
#define ANI_OK 0
#define ANI_ERR_BAD_ARG (-1)
#define ANI_ERR_UNSUPPORTED (-2)
#define ANI_ERR_CUDA (-3)

/* bits of the device status word (int32, written by kernels, never cleared by them) */
#define ANI_STATUS_NBR_OVERFLOW 1   /* an atom has more radial neighbours than nbr_cap   */
#define ANI_STATUS_ANG_OVERFLOW 2   /* an atom has more angular neighbours than ANI_MAX_ANG */
#define ANI_STATUS_CELL_TOO_SMALL 4 /* periodic cell thinner than the cutoff (neighbors.py:402-403) */
#define ANI_STATUS_PAIR_OVERFLOW 8  /* half neighbour list exceeds the caller's capacity */
#define ANI_VIRIAL_SLOTS 64         /* partial virial sums (ani_b200_aev_backward)          */
#define ANI_STATUS_OPERAND_RANGE 16 /* a value left the range of the half-precision GEMM operand pieces */
#define ANI_STATUS_INTERNAL 32      /* a device-side barrier / dependency wait timed out (never expected) */

#define ANI_MAX_ANG 96 /* angular neighbours (<= Rca) one central atom may have */

/* AEV constants; mirrors the CuaevComputer constructor (csrc/cuaev.cpp:247-278).       */
typedef struct ani_aev_params {
  float rcr, rca;            /* radial / angular cutoffs                                  */
  float eta_r, eta_a, zeta;  /* float32-rounded, as the reference's buffers hold them      */
  int32_t n_shf_r, n_shf_a, n_shf_z;
  int32_t num_species;
  int32_t cutoff_kind;       /* 0 = cosine (cutoffs.py:70-81), 1 = smooth (cutoffs.py:84-101) */
  float shf_r[ANI_MAX_SHFR];
  float shf_a[ANI_MAX_SHFA];
  float cos_z[ANI_MAX_SHFZ]; /* cos / sin of the angular sections ShfZ                     */
  float sin_z[ANI_MAX_SHFZ];
  /* internal column layout of the TILED AEV operand (ani_b200_aev_forward layout 1) and of the dE/dAEV rows the      */
  /* backward kernels read: the angular block starts ang_pad columns after the radial block, so that every element   */
  /* pair's 32 features fill exactly one 32-column GEMM block (ANI-2x: 7 x 16 radial columns + 16 = 128; water then   */
  /* has 5 live blocks instead of 8).  The padding columns are never written (zero) and the packed layer-1 weights    */
  /* hold zeros there.  0 = the reference's column order (always so for plain rows, layout 0).                        */
  int32_t ang_pad;
} ani_aev_params;

/* Device-resident description of the bucket grid, written by ani_b200_build_cells.     */
typedef struct ani_grid {
  float cell[9];   /* rows are lattice vectors (identity-like bounding box without PBC)  */
  float inv[9];    /* inverse: frac = (r - origin) @ inv                                  */
  float origin[3];
  int32_t dims[3]; /* buckets per lattice direction                                       */
  int32_t pbc;     /* 1 = periodic in all three directions                                */
  int32_t nbins;   /* real buckets; padding atoms live in bucket index nbins              */
  int32_t mode;    /* 0 = one conformer on a grid, 1 = batch, bucket == conformer         */
  int32_t n_per_conf;
  int32_t n_real;  /* number of non-padding atoms (== bin_start[nbins])                  */
} ani_grid;

int ani_b200_abi_version(void);

/* Format of the "tiled operand" matrices this build was compiled for (section 6):             */
/*   parts        16-bit pieces per value: 2 = IEEE half pieces of scale*x, 3 = bfloat16 pieces  */
/*   value_scale  power-of-two scale of AEV / activation operands (1 for bfloat16 pieces)        */
/*   grad_scale   power-of-two scale of gradient operands                                        */
/* No reference counterpart (the reference runs cuBLAS sgemm / TF32 on plain fp32 rows).         */
int ani_b200_operand_format(int32_t* parts, float* value_scale, float* grad_scale);
const char* ani_b200_error_string(int code);
/* Last CUDA error string seen by this library on the calling thread (for ANI_ERR_CUDA). */
const char* ani_b200_last_cuda_error(void);

/* ------------------------------------------------------------------------------------ */
/* 1. Bucket the atoms: wrap into the cell (PBC), assign buckets, stable counting sort.   */
/*    coords  [n_conf*n_per_conf*3] f32, species [n_conf*n_per_conf] i32 (-1 = padding)    */
/*    cell    device f32[9] (rows = lattice vectors) or NULL; pbc 0/1 (all directions)      */
/*    mode 0 requires n_conf == 1; mode 1 requires pbc == 0.                                */
/*    Outputs (all device):                                                                 */
/*      grid            ani_grid                                                            */
/*      bin_start       i32[max_bins+2]  exclusive scan of bucket populations               */
/*      sorted_orig     i32[n]           bucket-sorted position -> flat input index         */
/*      spos            f32[n*4]         wrapped x,y,z + species (int bits) in sorted order  */
/*      sbin            i32[n]           bucket of each sorted atom                         */
/*      orig_to_sorted  i32[n]           inverse of sorted_orig                             */
/*    Scratch: scratch_i32[3*n + max_bins + 2].                                             */
/*      bucket_ranges   f32[(max_bins-1)*27*8] or NULL: for every bucket the 27 neighbouring  */
/*                      buckets as {first atom, end atom, image code, -} + image shift vector   */
/*                      (mode 0 only; lets the AEV kernel skip the index / shift arithmetic)     */
int ani_b200_build_cells(const float* coords, const int32_t* species, int n_conf, int n_per_conf,
                         const float* cell, int pbc, int mode, float cutoff, int max_bins,
                         ani_grid* grid, int32_t* bin_start, int32_t* sorted_orig,
                         int32_t* orig_to_sorted, float* spos, int32_t* sbin, float* bucket_ranges,
                         int32_t* scratch_i32, int32_t* status, void* stream);

/* 2. Species-grouped row layout for the MLP: atoms lo..hi-1 (bucket-sorted positions,     */
/*    clipped to the real atoms) get rows grouped by species, every species block padded    */
/*    to a multiple of ANI_TILE_ROWS.                                                       */
/*      row_of      i32[n]        row of sorted atom i (undefined outside lo..hi-1)         */
/*      row_atom    i32[rows_cap] sorted atom of a row, -1 for padding rows                 */
/*      tile_species i32[rows_cap/ANI_TILE_ROWS]  species of each row tile, -1 = unused      */
/*      layout_info i32[16]: {n_tiles, n_rows, n_owned_atoms, 0, first row tile of species   */
/*                  0..S-1, total row tiles, ...}  (device-side tile lists of the GEMMs)      */
/*    Scratch: scratch_i32[(ceil(n/256)+2) * ANI_MAX_SPECIES + 64].                         */
int ani_b200_species_layout(const float* spos, const ani_grid* grid, int n, int lo, int hi,
                            int num_species, int rows_cap, int32_t* row_of, int32_t* row_atom,
                            int32_t* tile_species, int32_t* layout_info, int32_t* scratch_i32,
                            void* stream);

/* 2b. Active 32-column blocks of the AEV matrix: blocks[0] = count, blocks[1..] = ascending */
/*    block ids whose columns belong to an element / element pair present among the real      */
/*    atoms.  All other AEV columns are identically zero for every atom (and their gradient   */
/*    is never consumed), so the MLP may skip them.  blocks i32[ldx/32 + 3]: the last two words */
/*    hold the element-presence bit mask and a "mask changed since the previous call" flag      */
/*    (together: ani_b200_aev_forward's species_mask); scratch i32[1].                           */
int ani_b200_active_aev_blocks(const float* spos, const ani_grid* grid, int n, int num_species,
                               int n_shf_r, int angular_sub, int out_dim, int ldx, int ang_pad, int32_t* blocks,
                               int32_t* scratch_i32, void* stream);

/* 3. Fused neighbour search + AEV forward for sorted atoms lo..hi-1.                      */
/*      row_of     row of the output matrix for each sorted atom (species-grouped rows for   */
/*                 the fused engine, flat input index for the AEVComputer API)               */
/*      aev        layout 0: f32[rows][ldx], columns 0..out_dim-1 of the atom's row are      */
/*                 overwritten.  layout 1: the "tiled operand" form the MLP consumes          */
/*                 (see below; 6*rows_cap*ldx bytes, rows_cap % 128 == 0, ldx % 32 == 0)      */
/*      nbr_cnt    i32[n]; nbr_list i32[n*nbr_cap]: neighbours within Rcr of every processed  */
/*                 atom as (sorted index | image code << 26); kept for the backward pass      */
/*      bucket_ranges  output of ani_b200_build_cells or NULL (ranges are then derived on the   */
/*                 fly); species_mask: {bit per element present in the system, changed flag} or   */
/*                 NULL: angular blocks of absent element pairs are not rewritten while the       */
/*                 composition is unchanged (they hold zeros from the first call)                 */
/*      bucket_species  output of ani_b200_prepare_step or NULL (needs bucket_ranges): per bucket the offsets of   */
/*                 its species inside the (species-sorted) bucket, i32[nbins][8]; lets the kernel skip the pass that  */
/*                 counts the species of the ~370 staged candidates of a CTA                                          */
int ani_b200_aev_forward(const ani_aev_params* params, const ani_grid* grid,
                         const int32_t* bin_start, const float* spos, const int32_t* sbin,
                         const float* bucket_ranges, const int32_t* bucket_species, const int32_t* species_mask, int n, int lo,
                         int hi, const int32_t* row_of, float* aev, int ldx, int layout,
                         int32_t* nbr_cnt, int32_t* nbr_list, int nbr_cap, int32_t* status,
                         void* stream);

/* 4. AEV backward: grad_aev (same row layout as the forward output) -> dE/dcoords,         */
/*    accumulated (+=, float atomics) into grad_coords f32[n*3] in flat INPUT order.         */
/*    species_mask (as in the forward, or NULL): the gradient blocks of element pairs that   */
/*    do not occur in the system are not read (the block-sparse MLP backward leaves them     */
/*    unwritten).  max_elements (0 = num_species): how many distinct elements the caller      */
/*    expects in the system; it only sizes the kernel's shared-memory gradient table (higher   */
/*    occupancy for few-element systems) -- pairs beyond it are read from global memory, the   */
/*    result never depends on it.  virial (or NULL): f64[ANI_VIRIAL_SLOTS][9], zeroed by the     */
/*    caller; the kernel adds partial sums of W_ab = sum_pairs (dE/dDelta)_a Delta_b, the "f dot r" */
/*    virial of ase.py:164-168 (stress = sum over the slots / volume), row-major a, b.             */
int ani_b200_aev_backward(const ani_aev_params* params, const ani_grid* grid, const float* spos,
                          const int32_t* sorted_orig, const int32_t* species_mask, int n, int lo,
                          int hi, const int32_t* row_of, const float* grad_aev, int ldx,
                          const int32_t* nbr_cnt,
                          const int32_t* nbr_list, int nbr_cap, float* grad_coords,
                          int32_t* status, int max_elements, double* virial, void* stream);

/* 4b. The same AEV kernels fed by an externally supplied HALF pair list (the reference's    */
/*    Neighbors tuple; AEVComputer.compute_from_neighbors, aev/_computer.py:251-272 ->          */
/*    cuaev::run_with_half_nbrlist, csrc/aev.cu:1128-1208,1779-1866).  ani_b200_pairs_to_rows     */
/*    expands the list into per-atom rows (both directions): row_start i32[n+1], row_j i32[2P],  */
/*    row_d f32[2P][4] = (r_j - r_i, R); scratch i32[2n].  diff_vectors follow the reference:     */
/*    x[idx0] - x[idx1] + shift.  The *_rows entry points then take any `grid` whose n_real == n  */
/*    and an `spos` that only needs the species in .w (atoms in input order, padding = -1).       */
/*    Gradients go to the coordinates only, as in csrc/cuaev.cpp:158-163.                          */
int ani_b200_pairs_to_rows(const int64_t* idx0, const int64_t* idx1, const float* diff_vectors,
                           int64_t num_pairs, int n, int nbr_cap, int32_t* row_start,
                           int32_t* row_j, float* row_d, int32_t* scratch_i32, int32_t* status,
                           void* stream);
/* 4c. FULL neighbour list with ghost atoms, as MD engines hand it over (LAMMPS pair style, pmemd): replaces   */
/*    cuaev::run_with_full_nbrlist (csrc/cuaev.cpp:225-246, csrc/aev.cu:1048-1126,1868-1956;                      */
/*    aev/_computer.py:409-438).  coords f32[n_all][3] hold local AND ghost atoms (ghosts at their image          */
/*    positions, no cell), ilist i32[n_i] the atoms whose AEV is wanted, numneigh i32[n_i] their neighbour         */
/*    counts, jlist i32[sum numneigh] the neighbours of ilist[0], ilist[1], ... one after the other (built with    */
/*    cutoff + skin: entries beyond `cutoff` are screened out here).  Output: the per-atom rows of 4b              */
/*    (row_start i32[n_all+1], row_j / row_d with capacity sum(numneigh)); atoms not in ilist get empty rows, i.e.  */
/*    all-zero AEVs, as in the reference.  scratch i32[n_all + n_i + 1].  Feed the result to                         */
/*    ani_b200_aev_forward_rows / _backward_rows (gradients reach local and ghost coordinates alike).                */
int ani_b200_full_nbrlist_to_rows(const float* coords, int n_all, const int32_t* ilist, const int32_t* numneigh,
                                  const int32_t* jlist, int n_i, float cutoff, int nbr_cap, int32_t* row_start,
                                  int32_t* row_j, float* row_d, int32_t* scratch_i32, int32_t* status, void* stream);
int ani_b200_aev_forward_rows(const ani_aev_params* params, const ani_grid* grid, const float* spos,
                              const int32_t* row_start, const int32_t* row_j, const float* row_d,
                              int n, const int32_t* row_of, float* aev, int ldx, int layout,
                              int nbr_cap, int32_t* status, void* stream);
int ani_b200_aev_backward_rows(const ani_aev_params* params, const ani_grid* grid, const float* spos,
                               const int32_t* sorted_orig, const int32_t* row_start,
                               const int32_t* row_j, const float* row_d, int n, const int32_t* row_of,
                               const float* grad_aev, int ldx, int nbr_cap, float* grad_coords,
                               int32_t* status, void* stream);

/* 3c. Verlet-skin reuse of a bucket grid (neighbors.py:759-884, VerletCellList).  Build the grid  */
/*     with cutoff + skin (ani_b200_prepare_step / ani_b200_build_cells), then                      */
/*       mode 0  right after the build: remember the binned positions (ref_pos f32[n][4]) and the   */
/*               lattice vector that wrapped every atom into the cell (ref_shift f32[n][4]);        */
/*       mode 1  on later steps INSTEAD of a rebuild: spos = new coords + ref_shift in the same     */
/*               sorted order (every other output of the build stays valid), zero-fills             */
/*               zero_f32[0..count) like the fused preparation, and ORs into `moved` (i32[1],       */
/*               cleared by the caller) bit 0 if any atom is more than skin/2 from its binned        */
/*               position (the step is invalid), bit 1 if any is beyond 70 % of that (a hint to      */
/*               rebuild before the next step).                                                       */
/*     While bit 0 of `moved` stays 0 every pair within the true cutoff is still inside the 27 buckets around */
/*     an atom and the AEV kernels (which screen with the true cutoff and the current positions)    */
/*     give exactly the result of a rebuild; when it is raised the step must be redone after a      */
/*     rebuild.  aev_blocks (or NULL): the block list of the build, its "composition changed" flag  */
/*     is cleared in mode 1.                                                                          */
int ani_b200_verlet_positions(int mode, const float* coords, const ani_grid* grid,
                              const int32_t* sorted_orig, int n, float skin, float* spos, float* ref_pos,
                              float* ref_shift, int32_t* moved, float* zero_f32, int zero_f32_count,
                              int32_t* aev_blocks, int ldx, void* stream);

/* 3b. Fused per-step preparation: build_cells + species_layout + active_aev_blocks in ONE launch     */
/*     (a persistent grid with device-wide barriers between its five phases) instead of twelve       */
/*     (same outputs, same determinism; what the fused engine calls).                                 */
/*     Also zero-fills zero_f32[0..count) (the force accumulator) and zero_f64[0..count) (the      */
/*     conformer energies) so that no separate memset launches are needed.                          */
/*     bucket_species (or NULL): i32[max_bins][8], per bucket the offset of its first atom of species >= s */
/*     (buckets are species-sorted), consumed by ani_b200_aev_forward.                               */
/*     scratch_i32: 3 n + max_bins + 4 + (ceil((hi-lo)/256) + 2) * ANI_MAX_SPECIES + 32 ints, ZERO at           */
/*     allocation (two of them are the state of the device-wide barrier of the single-launch preparation).     */
int ani_b200_prepare_step(const float* coords, const int32_t* species, int n_conf, int n_per_conf,
                          const float* cell, int pbc, int mode, float cutoff, int max_bins, ani_grid* grid,
                          int32_t* bin_start, int32_t* sorted_orig, int32_t* orig_to_sorted, float* spos,
                          int32_t* sbin, float* bucket_ranges, int lo, int hi, int num_species, int rows_cap,
                          int32_t* row_of, int32_t* row_atom, int32_t* tile_species, int32_t* layout_info,
                          int n_shf_r, int angular_sub, int out_dim, int ldx, int ang_pad, int32_t* aev_blocks,
                          float* zero_f32, int zero_f32_count, double* zero_f64, int zero_f64_count,
                          int32_t* bucket_species, int32_t* scratch_i32, int32_t* status, void* stream);

/* Timing experiments only: the first 4 CTAs of the next `launches` tensor-core GEMM launches    */
/* write clock64 stamps [launch][cta 4][tile 8][role 3: producer, MMA, epilogue][4] into buf       */
/* (device memory, launches*384 int64).  NULL switches it off.  No reference counterpart.           */
int ani_b200_debug_gemm_trace(long long* buf, int launches);

/* 5. Reference-format half neighbour list (neighbors.py:13-18) from the bucket grid.       */
/*    Two calls: count (fills pair_start i32[n+1], exclusive scan, total in pair_start[n]),  */
/*    then fill with capacity `cap` pairs.  indices are flat INPUT indices, idx0 < idx1       */
/*    except for self-image pairs; diff = x[idx0] - x[idx1] + shift (neighbors.py:107-111).   */
int ani_b200_half_neighbor_count(const ani_grid* grid, const int32_t* bin_start, const float* spos,
                                 const int32_t* sbin, const int32_t* sorted_orig, int n,
                                 float cutoff, int32_t* pair_start, void* stream);
int ani_b200_half_neighbor_fill(const ani_grid* grid, const int32_t* bin_start, const float* spos,
                                const int32_t* sbin, const int32_t* sorted_orig, int n, float cutoff,
                                const int32_t* pair_start, int64_t cap, int64_t* idx0, int64_t* idx1,
                                float* distances, float* diff_vectors, int32_t* status, void* stream);

/* 6. Ensemble MLP forward + backward-to-input on the species-grouped AEV matrix.           */
/*    Layer widths: in -> h1 -> h2 -> h3 -> 1, CELU(alpha) after the three hidden layers.    */
/*    "Tiled operand" layout (both GEMM operands; fp32 accuracy on the tensor cores from 16-bit    */
/*    pieces, see ani_b200_operand_format): every value x of an operand with power-of-two scale s   */
/*    is stored as P pieces with s*x = p1 + ... + pP, each rounded to nearest:                       */
/*      P = 2 IEEE half pieces (default build; 4 B/element; s = 64 for AEVs/activations, 4096 for    */
/*            gradients, ani_mlp_species::w_scale for weights; |s*x| must stay below 65504, else     */
/*            ANI_STATUS_OPERAND_RANGE is raised and the results are inf/NaN),                       */
/*      P = 3 bfloat16 pieces (-DANI_OPND_FP16X2=0; 6 B/element; s = 1).                             */
/*    * A operand / activation matrix [rows][cols] (rows % 128 == 0, cols % 32 == 0):                */
/*        [row tile of 128][32-column block][p1: 128 rows x 64 B | p2 (| p3)]    (16 / 24 KB blocks) */
/*    * B operand of a layer GEMM  C[rows, N] = A[rows, K] x W  (W given as B[N][K], N % 32 == 0,  */
/*      K padded to a multiple of 32 with zeros):                                                  */
/*        [member][n tile (256 rows, the last one shorter)][32-column block][p1 bn x 64 B | p2 (| p3)] */
/*    In both, every 8-row x 64-byte group is in the tcgen05 SWIZZLE_64B order (16-byte chunk c    */
/*    of row r sits at chunk position c ^ ((r >> 1) & 3)), i.e. exactly the shared-memory image    */
/*    a K-major UMMA descriptor expects: one K-block of one tile is a contiguous byte range        */
/*    that a single cp.async.bulk (TMA) moves into shared memory.  Hidden widths that are not       */
/*    multiples of 32 are zero-padded by the packer (zero weights and biases: CELU(0) = 0).         */
typedef struct ani_mlp_species {
  int32_t h1, h2, h3, pad_;
  float w_scale[4];  /* [0..2]: power-of-two scale the packer multiplied W1, W2, W3 by (fp16 pieces) */
  const float* b1;   /* [M*h1]                                                                  */
  const float* b2;   /* [M*h2]                                                                  */
  const float* b3;   /* [M*h3]                                                                  */
  const float* w4;   /* [M][h3]                                                                 */
  const float* b4;   /* [M]                                                                     */
  const void* t_f1;  /* forward  layer 1: per member B = W1_m [h1][in_dim -> ldx]               */
  const void* t_f2;  /* forward  layer 2: per member B = W2_m [h2][h1]                          */
  const void* t_f3;  /* forward  layer 3: per member B = W3_m [h3][h2]                          */
  const void* t_b3;  /* backward layer 3: per member B = W3_m^T [h2][h3]                        */
  const void* t_b2;  /* backward layer 2: per member B = W2_m^T [h1][h2]                        */
  const void* t_b1;  /* backward layer 1: B = W1^T [ldx][M*h1]                                  */
} ani_mlp_species;

typedef struct ani_mlp_model {
  int32_t num_species, num_members, in_dim, ldx;
  int32_t h1_max, h2_max, h3_max, pad_;
  float celu_alpha;
  float member_scale[ANI_MAX_MEMBERS]; /* d(output)/d(member energy): 1/M_active or 0       */
  ani_mlp_species sp[ANI_MAX_SPECIES];
  /* optional device scratch, sum over the species of ldx * (M * h1 / 32) * 2 * P * 32 bytes (the size of the t_b1   */
  /* operands together), or NULL: every step gathers the LIVE column blocks of the layer-1 backward operands into   */
  /* it (ani_b200_zero_live_blocks / ani_b200_mlp_step / ani_b200_mlp_backward), so that the GEMM moves one         */
  /* K-block of them with one bulk copy.  No state is carried between steps; one step at a time per model.          */
  void* b1_compact;
} ani_mlp_model;

/* 6a. Model-pack time: plain fp32 weights -> the tiled B operand above (one launch per operand; `batch`   */
/*     operands of the same shape, e.g. the members of an ensemble, src/dst `*_batch_stride` elements/bytes     */
/*     apart).  src is [n][ld_src] (B[n][k] = src[n][k]) or, with transpose != 0, [k][ld_src] (B[n][k] =       */
/*     src[k][n]: the backward operands are the transposed weights); n % 32 == 0; K is zero-padded to a        */
/*     multiple of 32; every value is multiplied by the power-of-two `scale` first.                             */
/*     dst: batch * n * ceil32(k) * 2 * P bytes.  Replaces BmmLinear.__init__ (nn/_infer.py:171-203), the       */
/*     reference's own inference-time re-layout of the weights.                                                 */
int ani_b200_pack_b_operand(const float* src, int n, int k, int ld_src, int transpose, float scale, int batch,
                            long long src_batch_stride, void* dst, long long dst_batch_stride, void* stream);

/*    x            tiled operand, in: AEVs (ani_b200_aev_forward layout 1), 2*P*rows_cap*ldx bytes */
/*    dx           f32[rows_cap][ldx] plain rows, out: dE/dAEV (may be NULL if !want_backward)  */
/*    row_atom / layout_info: outputs of ani_b200_species_layout                                */
/*    aev_blocks   output of ani_b200_active_aev_blocks or NULL (= every column is live).       */
/*                 With a block list, layer 1 skips the dead K-blocks and dE/dAEV is written     */
/*                 only for the live column blocks (the others keep their previous content).     */
/*    act1/2/3     tiled operands, 2*P*rows_cap*M*h{1,2,3}_max bytes (activations, then gradients) */
/*    e_member     f32[M][rows_cap]     per-member atomic energies                               */
/*    status       i32[1] device word, ANI_STATUS_OPERAND_RANGE is OR-ed in (may be NULL)        */
int ani_b200_mlp_forward_backward(const ani_mlp_model* model, const void* x, float* dx, int rows_cap,
                                  const int32_t* row_atom, const int32_t* layout_info,
                                  const int32_t* aev_blocks, void* act1, void* act2, void* act3,
                                  float* e_member, int want_backward, int32_t* status, void* stream);

/*    The same work as two calls, so that a caller can run independent work beside the backward      */
/*    GEMMs (engine.py: ani_b200_reduce_energies only needs e_member, i.e. the forward half) and      */
/*    zero dE/dAEV ahead of time on another stream:                                                    */
/*      ani_b200_mlp_forward       layers 1-3 + final layer + gradient seed (act3)                    */
/*      ani_b200_zero_live_blocks  dx[rows][live column blocks] = 0 (the layer-1 backward accumulates  */
/*                                 the members into dx; only needed when num_members > 1)              */
/*      ani_b200_mlp_backward      the three backward-to-input GEMMs; dx_zeroed != 0: the caller has   */
/*                                 already run ani_b200_zero_live_blocks for this step                 */
int ani_b200_mlp_forward(const ani_mlp_model* model, const void* x, int rows_cap, const int32_t* row_atom,
                         const int32_t* layout_info, const int32_t* aev_blocks, void* act1, void* act2,
                         void* act3, float* e_member, int want_backward, int32_t* status, void* stream);
int ani_b200_zero_live_blocks(const ani_mlp_model* model, float* dx, const int32_t* layout_info,
                              const int32_t* aev_blocks, void* stream);
int ani_b200_mlp_backward(const ani_mlp_model* model, float* dx, int rows_cap, const int32_t* row_atom,
                          const int32_t* layout_info, const int32_t* aev_blocks, void* act1, void* act2,
                          void* act3, int dx_zeroed, int32_t* status, void* stream);

/*    The same six GEMMs as ONE persistent launch (csrc/gemm_fused.cuh): the (layer, row tile, member, column      */
/*    tile) units form one list and the launch boundaries are replaced by data-flow waits on per-(layer, row tile)   */
/*    completion counters -- no ramp / tail per layer, one tile-count quantisation for the whole step, and at small   */
/*    row counts (multi-GPU shards) no per-launch floor.  sync_i32: 6 * (rows_cap / 128) ints of scratch (zeroed by    */
/*    the call).  Same arguments and results as ani_b200_mlp_forward_backward otherwise.  want_backward == 2:          */
/*    PER-MEMBER gradients (arch.py:403-436, members_forces): dx is f32[M][rows_cap][ldx] and member m's slab receives   */
/*    d(member_scale[m] * e_m)/dAEV by plain stores (no sum over the members, no zero-fill needed).                      */
/*    ani_b200_mlp_step runs a step as ani_b200_mlp_step_windows(model, rows_cap) launches of the data-flow kernel, */
/*    one per window of the row tiles (all six phases of a window, then the next), sized so that a window's         */
/*    activations stay in the L2 between the phase that writes them and the phases that read them.                  */
int ani_b200_mlp_step_windows(const ani_mlp_model* model, int rows_cap);
/*    Which kernel ani_b200_mlp_step launches for this model and row capacity: 0 the data-flow launch, 1 independent */
/*    chains (ANI_B200_MLP_CHAIN=1), 2 resident chains (csrc/gemm_resident.cuh: a CTA runs one (row tile, member)     */
/*    chain at a time with its activations and gradients in shared memory; the default where its shared-memory plan  */
/*    fits and there are at most 8 chains per SM, ANI_B200_MLP_RESIDENT=0 / 1: never / whatever the length).          */
int ani_b200_mlp_step_kernel(const ani_mlp_model* model, int rows_cap);
/*    The shared-memory plan of the resident-chain kernel, bytes: out[0] resident image, out[1] weight ring of        */
/*    layers 2-6, out[2] layer-1 ring (over both), out[3] dynamic shared memory available; out[4] 1 if it fits.       */
int ani_b200_mlp_resident_plan(const ani_mlp_model* model, int32_t* out);
int ani_b200_mlp_step(const ani_mlp_model* model, const void* x, float* dx, int rows_cap, const int32_t* row_atom,
                      const int32_t* layout_info, const int32_t* aev_blocks, void* act1, void* act2, void* act3,
                      float* e_member, int want_backward, int32_t* sync_i32, int32_t* status, void* stream);

/* 7. Scatter per-member atomic energies back to input order and reduce per conformer.      */
/*      atomic_out f32[n] (mean over active members, 0 for padding; flat input order)         */
/*      member_atomic_out f32[M][n] or NULL                                                    */
/*      energies_out f64[n_conf]  NN energy + self energies (sae f64[num_species] or NULL)     */
/*    Only atoms whose sorted position is in lo..hi-1 contribute (others give 0), so the     */
/*    per-rank results of a sharded run add up to the full answer.                            */
int ani_b200_reduce_energies(const ani_mlp_model* model, const float* e_member, int rows_cap,
                             const int32_t* row_of, const int32_t* orig_to_sorted,
                             const int32_t* species, int n, int lo, int hi, int n_conf,
                             int n_per_conf, const double* sae, float* atomic_out,
                             float* member_atomic_out, double* energies_out, void* stream);

/* 8. Multi-GPU: one-shot all-reduce of the per-rank partial forces / energies over NVLink peer memory.   */
/*    The path shards by central atom (one process per GPU); every rank accumulates dE_owned/dx_j into a      */
/*    full-length f32[n_f32] buffer and its share of the conformer energies into f64[n_f64].  Those partial     */
/*    buffers live in CUDA-IPC memory owned by the communicator (the ONE place where this library allocates:    */
/*    IPC-exportable memory must come from cudaMalloc) and are mapped by every peer; ani_b200_comm_allreduce     */
/*    launches ONE kernel: flag barrier in peer memory, every rank sums the W partials in rank order (bitwise      */
/*    identical totals everywhere) into its own out buffers, flag barrier.  Graph-capturable; epochs advance on     */
/*    the device.  The reference has no collective (SURVEY.md 2.1) -- this replaces the NCCL all-reduce of         */
/*    round 1 (parallel.py).  Set-up: create on every rank, exchange the 64-byte handles by any host channel        */
/*    (torch.distributed all_gather here), connect with the W handles in rank order.  world <= 8, one node.          */
/*    error_word (device i32): raised by the kernel if a peer does not arrive within ~10 s (no hang).               */
int ani_b200_comm_create(int rank, int world, long long n_f32, long long n_f64, void** comm_out);
int ani_b200_comm_handle(void* comm, void* handle64);
int ani_b200_comm_connect(void* comm, const void* handles);
int ani_b200_comm_buffers(void* comm, float** partial_f32, double** partial_f64, int32_t** error_word);
int ani_b200_comm_allreduce(void* comm, float* out_f32, double* out_f64, void* stream);
int ani_b200_comm_destroy(void* comm);

#ifdef __cplusplus
}
#endif
#endif /* ANI_B200_H */
