/*
 * dmpnn.h -- C ABI of libdmpnn_sm100.so, the B200 (sm_100a) D-MPNN message-passing engine.
 *
 * The reference (chemprop v2.3.1) has no FFI on this path: the hot path is ~150 lines of
 * Python dispatching stock ATen ops.  This header is therefore the boundary a maintainer
 * would bind (ctypes) from the reference's module layer; each entry point names the
 * reference code (file:line, relative to the chemprop repo root) it replaces.
 *
 * Conventions
 *  - Plain C symbols; raw device pointers; int64_t sizes; `stream` is a cudaStream_t passed
 *    as void* (torch.cuda.current_stream().cuda_stream).  No torch types.
 *  - The library never allocates, frees or synchronises; all buffers (outputs, saved
 *    activations, workspaces) are owned by the caller.  Launches are asynchronous on `stream`.
 *  - Every function returns 0 on success, <0 on error; dmpnn_last_error() gives the
 *    thread-local message.
 *  - "Hidden" matrices (edge / atom hidden states) are row-major with a row stride `ld`
 *    given in ELEMENTS; their element type is `dmpnn_dtype_t` (f32 or bf16).  Inputs V, E and
 *    all weights / weight gradients are f32.
 *  - Internal edge order: the engine keeps edge hidden states sorted by destination atom
 *    (stable), so the in-edges of atom v are the contiguous rows [rowptr[v], rowptr[v+1]).
 *    `perm[row]` is the caller's edge id of an internal row; outputs of the path are atom- or
 *    molecule-level, so this order never leaks out.
 */
#ifndef DMPNN_H_
#define DMPNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMPNN_VERSION 100 /* 0.1.0 */

typedef enum { DMPNN_F32 = 0, DMPNN_BF16 = 1 } dmpnn_dtype_t;

/* Activations of chemprop/nn/utils.py:11-55 that the engine fuses (PReLU / arbitrary modules
 * are handled by the Python host as an unfused composition). */
typedef enum {
  DMPNN_ACT_NONE = 0,
  DMPNN_ACT_RELU = 1,
  DMPNN_ACT_LEAKYRELU = 2, /* slope = act_param (reference: 0.1) */
  DMPNN_ACT_TANH = 3,
  DMPNN_ACT_ELU = 4 /* alpha = act_param (reference: 1.0) */
} dmpnn_act_t;

/* segment scaling: none; divide by the constant `scale` (NormAggregation, agg.py:112-113);
 * divide by the segment's row count (MeanAggregation, agg.py:73-78; empty segment -> 0). */
typedef enum { DMPNN_SCALE_NONE = 0, DMPNN_SCALE_DIV_CONST = 1, DMPNN_SCALE_INV_COUNT = 2 } dmpnn_scale_t;

/* Layout meta words written by dmpnn_layout_build (int32 each). */
enum {
  DMPNN_META_N_TILES = 0,      /* number of molecule-aligned tiles                              */
  DMPNN_META_FLAGS = 1,        /* bit set below                                                 */
  DMPNN_META_MAX_INDEG = 2,    /* max in-degree of any atom                                     */
  DMPNN_META_MAX_TILE_ROWS = 3,/* largest tile (edge rows); >128 => some molecule is oversized  */
  DMPNN_META_MAX_TILE_ATOMS = 4,
  DMPNN_META_WORDS = 8
};
enum {
  DMPNN_FLAG_REV_INVOLUTION = 1, /* rev[rev[e]]==e, src[rev e]==dst[e], dst[rev e]==src[e]      */
  DMPNN_FLAG_BATCH_SORTED = 2,   /* batch non-decreasing and every edge intra-molecule          */
  DMPNN_FLAG_INDEX_IN_RANGE = 4  /* all indices within [0,V) / [0,E) / [0,B)                    */
};

int dmpnn_version(void);
const char* dmpnn_last_error(void);
/* 1 if a CUDA device of compute capability 10.x is current, else 0 (never throws). */
int dmpnn_device_ok(void);
/* Number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
long long dmpnn_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * Host-side collate.  Replaces BatchMolGraph.__post_init__ (chemprop/data/collate.py:37-62):
 * concatenates per-molecule arrays and offsets edge_index / rev_edge_index; produces the same
 * five public arrays (V, E f32; edge_index 2xE, rev_edge_index E, batch V -- all int64).
 * CPU code (the reference runs this in DataLoader worker processes).
 * `n_atoms[i]`, `n_edges[i]` give molecule sizes; `V_ptrs[i]` etc. point at that molecule's
 * arrays (V: n_atoms x d_v f32; E: n_edges x d_e f32; edge_index: 2 x n_edges int64 row-major;
 * rev: n_edges int64).
 * ------------------------------------------------------------------------------------- */
int dmpnn_collate_host(int64_t n_mols, const int64_t* n_atoms, const int64_t* n_edges,
                       const float* const* V_ptrs, const float* const* E_ptrs,
                       const int64_t* const* edge_index_ptrs, const int64_t* const* rev_ptrs,
                       int64_t d_v, int64_t d_e,
                       float* V_out, float* E_out, int64_t* edge_index_out /*2 x E_tot*/,
                       int64_t* rev_out, int64_t* batch_out);

/* The same batch in the compact transfer format (bf16 features, round-to-nearest-even; int32 indices): what
 * BatchMolGraph(transfer_dtype=bfloat16) copies host -> device instead of the f32 / int64 tensors.  The bf16 tier
 * rounds V / E to bf16 when it assembles its GEMM operands, so its results do not change.  Fails (< 0) when the
 * batch does not fit int32 indices. */
int dmpnn_collate_host_compact(int64_t n_mols, const int64_t* n_atoms, const int64_t* n_edges,
                               const float* const* V_ptrs, const float* const* E_ptrs,
                               const int64_t* const* edge_index_ptrs, const int64_t* const* rev_ptrs,
                               int64_t d_v, int64_t d_e,
                               uint16_t* V_out, uint16_t* E_out, int32_t* edge_index_out /*2 x E_tot*/,
                               int32_t* rev_out, int32_t* batch_out);

/* ---------------------------------------------------------------------------------------
 * Packed dataset (SURVEY.md 8f-1): all molecules of a data set in flat arrays -- V_all (sum V x d_v f32), E_all
 * (sum E x d_e f32), molecule-LOCAL edge_index (2 x sum E, int32) and rev_edge_index (sum E, int32), atom_ptr /
 * edge_ptr (n + 1, int64) -- on the host or resident in HBM.  A batch for the molecule ids `ids` is one gather:
 * replaces `[dataset[i] for i in ids]` + collate_batch (chemprop/data/datasets.py:222-244, collate.py:37-97) and,
 * for the device-resident form, the host -> device copy of the batch.
 *   dmpnn_dataset_batch_meta_host  output offsets of the selected molecules (out_atom_ptr / out_edge_ptr, n_sel + 1
 *                                  each) and the batch's layout meta words in O(n_sel) from per-molecule sizes
 *                                  (`mol_max_indeg`: max in-degree of each molecule; molecules are validated once,
 *                                  when the data set is packed, so all three flags are set).  CPU code.
 *   dmpnn_dataset_gather_host      the five public BatchMolGraph arrays (f32 / int64; any of V_out, E_out, ei_out +
 *                                  rev_out, batch_out may be NULL to skip it) and, when the five compact pointers
 *                                  are given, the bf16 / int32 transfer copy, in one pass, the selection split over host threads.
 *                                  CPU code.
 *   dmpnn_dataset_gather           the same five arrays on the device: one block per selected molecule, contiguous
 *                                  row copies (16 / 8 / 4-byte accesses by feature width), indices offset on the fly.
 *                                  All pointers are device pointers; ids / out_*_ptr are what the host computed with
 *                                  dmpnn_dataset_batch_meta_host and uploaded (24 bytes per molecule).
 * ------------------------------------------------------------------------------------- */
int dmpnn_dataset_batch_meta_host(int64_t n_sel, const int64_t* ids, int64_t n_total, const int64_t* atom_ptr,
                                  const int64_t* edge_ptr, const int32_t* mol_max_indeg, int64_t* out_atom_ptr,
                                  int64_t* out_edge_ptr, int32_t* meta /*DMPNN_META_WORDS*/);
int dmpnn_dataset_gather_host(int64_t n_sel, const int64_t* ids, const int64_t* out_atom_ptr, const int64_t* out_edge_ptr,
                              const int64_t* atom_ptr, const int64_t* edge_ptr, const float* V_all, const float* E_all,
                              const int32_t* ei_local, const int32_t* rev_local, int64_t E_all_total, int64_t d_v,
                              int64_t d_e, float* V_out, float* E_out, int64_t* ei_out /*2 x E_out*/, int64_t* rev_out,
                              int64_t* batch_out, uint16_t* Vb_out, uint16_t* Eb_out, int32_t* ei32_out,
                              int32_t* rev32_out, int32_t* batch32_out, int n_threads /* <= 0: automatic */);
int dmpnn_dataset_gather(const int64_t* ids, const int64_t* out_atom_ptr, const int64_t* out_edge_ptr, int64_t n_sel,
                         const int64_t* atom_ptr, const int64_t* edge_ptr, const float* V_all, const float* E_all,
                         const int32_t* ei_local, const int32_t* rev_local, int64_t E_all_total, int64_t d_v, int64_t d_e,
                         float* V_out, float* E_out, int64_t* ei_out /*2 x E_out_total*/, int64_t* rev_out,
                         int64_t* batch_out, int64_t E_out_total, void* stream);

/* Dropout application (chemprop/nn/message_passing/base.py:139, :182; nn.Dropout): OUT[i] = X[i] * M[i] * scale over a flat
 * contiguous buffer of n elements of type `dtype` (a hidden matrix with its padding columns), M a {0, 1} keep mask of the same
 * element type drawn by the caller's RNG (torch's Philox stream, so `torch.manual_seed` governs it as in the reference),
 * scale = 1 / (1 - p) applied in f32 with one rounding.  In place allowed (OUT == X). */
int dmpnn_scale_mask(const void* X, const void* M, void* OUT, int dtype, int64_t n, float scale, void* stream);

/* Loader-side molecule order for full tiles: a permutation of the batch's molecules (best-fit-decreasing bin packing of
 * their edge counts into the 128-row / 128-atom tiles of dmpnn_layout_build) under which the greedy tile packing of
 * CONSECUTIVE molecules comes out ~0.94 full instead of ~0.81 for ~25-atom molecules in arrival order.  The order of
 * the molecules inside a batch is the loader's to choose (the reference shuffles it every epoch, samplers.py:19-23);
 * tiles are always derived exactly from the final order, so this is a performance heuristic only.  CPU code. */
int dmpnn_tile_pack_order(int64_t n, const int64_t* n_atoms, const int64_t* n_edges, int64_t* order_out /*n*/);

/* Layout meta words of a batch computed on the HOST (same DMPNN_META_* words dmpnn_layout_build writes on the
 * device): validity flags, max in-degree, and the tile count / largest tile of the greedy molecule-aligned packing.
 * A loader calls it next to the collate (the batch's int64 index arrays are in host memory there), so that the
 * training step never reads `meta` back from the GPU: no host <-> device synchronisation inside the step.  The
 * reference has the same kind of per-batch sync in agg.py:75 (`batch.max().int() + 1`).  Bit-exact w.r.t.
 * oracle/layout_np.py; for an invalid batch only DMPNN_META_FLAGS is meaningful.  CPU code. */
int dmpnn_batch_meta_host(const int64_t* edge_index /*2 x E*/, const int64_t* rev_edge_index, const int64_t* batch,
                          int64_t V, int64_t E, int64_t B, int32_t* meta /*DMPNN_META_WORDS*/);

/* ---------------------------------------------------------------------------------------
 * Device layout build.  Consumes the reference's BatchMolGraph index tensors
 * (chemprop/data/collate.py:24-33: edge_index int64 2xE, rev_edge_index int64 E, batch int64 V)
 * and produces the engine's int32 layout: the stable sort of edges by destination atom
 * (perm / inv_perm / rowptr), per-row src / dst / rev (internal row ids), molecule atom/row
 * offsets, and a table of molecule-aligned tiles holding <=128 edge rows and <=128 atoms each
 * (a molecule larger than that gets a tile of its own; see DMPNN_META_MAX_TILE_*).
 * This replaces the index materialisation in chemprop/nn/message_passing/mixins.py:12
 * (`edge_index[1].unsqueeze(1).repeat(1, h)`) and chemprop/nn/agg.py:74-75.
 * Integer outputs are bit-exact w.r.t. oracle/layout_np.py.
 * ------------------------------------------------------------------------------------- */
int dmpnn_layout_workspace_bytes(int64_t V, int64_t E, int64_t B, size_t* bytes);
int dmpnn_layout_build(const int64_t* edge_index, const int64_t* rev_edge_index, const int64_t* batch,
                       int64_t V, int64_t E, int64_t B,
                       int32_t* perm /*E*/, int32_t* inv_perm /*E*/, int32_t* rowptr /*V+1*/,
                       int32_t* src_row /*E*/, int32_t* dst_row /*E*/, int32_t* rev_row /*E*/,
                       int32_t* mol_atom_ptr /*B+1*/, int32_t* mol_row_ptr /*B+1*/,
                       int32_t* tile_mol_ptr /*B+1, first n_tiles+1 valid*/,
                       int32_t* tile_row_ptr /*B+1: first internal row of each tile (+ sentinel)*/,
                       int32_t* tile_atom_ptr /*B+1: first atom of each tile (+ sentinel)*/,
                       int32_t* meta /*DMPNN_META_WORDS*/,
                       void* workspace, void* stream);

/* Segment offsets of a sorted int64 index (the `batch` argument of Aggregation.forward,
 * chemprop/nn/agg.py:39-59): ptr[b] = first i with index[i] >= b, ptr[n_seg] = n.  `status`
 * (1 int32, device) is set non-zero if index is not non-decreasing or leaves [0, n_seg). */
int dmpnn_sorted_index_to_ptr(const int64_t* index, int64_t n, int64_t n_seg, int32_t* ptr,
                              int32_t* status, void* stream);

/* ---------------------------------------------------------------------------------------
 * Generic fused linear:  C[cr(r), 0:N] = act( [X1[i1(r)] || X2[i2(r)]] . W^T + bias + R[r] )
 * for r in [0,R).  W is the nn.Linear weight, f32 row-major N x (K1+K2), row stride ldw.
 * X1 / X2: f32 or hidden dtype (per *_dtype); idx1 / idx2 optional int32 row gathers (NULL =
 * identity); K2 may be 0.  bias (f32, N) and residual R (hidden dtype, ldr) optional (NULL).
 * Columns [N, ldc_pad) of C are zero-filled (ldc_pad <= ldc), keeping row padding clean.
 * Covers: W_i initialise (mixins.py:8-9, :22-23), W_h update (base.py:135-141), W_o finalize
 * (base.py:180-182) and the dX = dY.W GEMMs of their autograd mirror.
 * fp32-accurate SIMT path (no tensor cores): this is the <=1e-5 tier and the fallback.
 * ------------------------------------------------------------------------------------- */
int dmpnn_linear_fwd(const void* X1, int x1_dtype, int64_t ld1, const int32_t* idx1, int64_t K1,
                     const void* X2, int x2_dtype, int64_t ld2, const int32_t* idx2, int64_t K2,
                     const float* W, int64_t ldw, const float* bias,
                     const void* Rres, int r_dtype, int64_t ldr,
                     int act, float act_param,
                     void* C, int c_dtype, int64_t ldc, int64_t ldc_pad,
                     int64_t R, int64_t N, void* stream);

/* Weight gradient: dW[n, 0:K1+K2] (+)= sum_r dY[r,n] * [X1[i1(r)] || X2[i2(r)]][k];
 * optional dbias[n] (+)= sum_r dY[r,n].  Two-pass deterministic reduction through
 * `workspace` (dmpnn_linear_wgrad_workspace_bytes).  accumulate!=0 adds into dW / dbias. */
int dmpnn_linear_wgrad_workspace_bytes(int64_t R, int64_t N, int64_t K, size_t* bytes);
int dmpnn_linear_wgrad(const void* dY, int dy_dtype, int64_t lddy,
                       const void* X1, int x1_dtype, int64_t ld1, const int32_t* idx1, int64_t K1,
                       const void* X2, int x2_dtype, int64_t ld2, const int32_t* idx2, int64_t K2,
                       float* dW, int64_t lddw, float* dbias, int accumulate,
                       int64_t R, int64_t N, void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------
 * Segmented row sum:  Y[s, 0:C] = scale(s) * sum_{r in [ptr[s], ptr[s+1])} f(X[idx(r), 0:C]).
 * f = activation `act` applied on load (ACT_NONE = identity).  Covers the final atom
 * scatter-sum (base.py:208-211; segments = atoms over dst-sorted rows), the neighbour sum of
 * the atom-granular AtomMessagePassing (mixins.py:25-30), and Mean/Sum/Norm aggregation
 * (agg.py:73-78, 90-95, 112-113; segments = molecules; divide by count / nothing / norm).
 * Empty segments give zero rows (agg.py:44-45).  Accumulates in f32, deterministic order.
 * ------------------------------------------------------------------------------------- */
int dmpnn_segment_sum(const void* X, int x_dtype, int64_t ldx, const int32_t* idx,
                      const int32_t* ptr, int64_t n_seg, int64_t C,
                      int act, float act_param, int scale_mode, float scale,
                      void* Y, int y_dtype, int64_t ldy, int64_t ldy_pad, void* stream);

/* Row broadcast (autograd mirror of segment_sum with identity f):
 * Y[r, 0:C] = scale(seg(r)) * G[seg_of_row[r], 0:C]; for SCALE_INV_COUNT, `ptr` gives counts.
 * n_seg > 0 (with ptr): the rows of segment s are exactly [ptr[s], ptr[s+1]) (the segment_sum convention,
 * ptr[n_seg] == R); the kernel then walks segments -- one scaled row of G held in registers, streamed to its
 * rows -- and never reads seg_of_row.  n_seg == 0: per-row lookup through seg_of_row. */
int dmpnn_segment_bcast(const void* G, int g_dtype, int64_t ldg, const int32_t* seg_of_row,
                        const int32_t* ptr, int64_t n_seg, int64_t R, int64_t C, int scale_mode, float scale,
                        void* Y, int y_dtype, int64_t ldy, void* stream);

/* ---------------------------------------------------------------------------------------
 * Bond message (mixins.py:11-18):  M[e] = sum_{e': dst(e')=src(e)} H[e'] - H[rev(e)], computed
 * per atom v over its in-edge rows e'_1..e'_d:  s = sum_i f(X[rd(e'_i)]);
 * OUT[wr(e'_i)] = s - f(X[rd(e'_i)])  with (rd, wr) = (identity, rev) when permute_on_read==0
 * (forward: OUT = M) and (rev, identity) when permute_on_read!=0 (autograd mirror:
 * dH[e] = sum_{src(e'')=dst(e)} dM[e''] - dM[rev(e)]).  Requires DMPNN_FLAG_REV_INVOLUTION.
 * f = `act` on load (used at depth step 1 where H^0 = tau(H_0), base.py:200).
 * ------------------------------------------------------------------------------------- */
int dmpnn_bond_message(const void* X, int x_dtype, int64_t ldx,
                       const int32_t* rowptr, const int32_t* rev_row, int64_t V, int64_t C,
                       int act, float act_param, int permute_on_read,
                       void* OUT, int out_dtype, int64_t ldo, void* stream);

/* Autograd mirror of the message with tau' fused: OUT[r] = (sum_{r' in seg(dst r)} X[rev r'] - X[rev r]) * tau'(Y[r])
 * (= dZ^{t-1} from dM^t and the stored H^{t-1}); one dtype for X / Y / OUT; C % 4 == 0, 4-element aligned. */
int dmpnn_bond_message_bwd_masked(const void* X, int dtype, int64_t ldx, const int32_t* rowptr, const int32_t* rev_row,
                                  int64_t V, int64_t C, const void* Yact, int64_t ldy, int act, float act_param,
                                  void* OUT, int64_t ldo, void* stream);
/* OUT[r] = sum_{k<n_z} Z_k[r] + G[r] * tau'(Ypre[r])  (tau' from the PRE-activation; G may be NULL): the total dH_0 of
 * base.py:135-141's autograd mirror in one pass.  Z: host array of <= 8 device pointers sharing ldz / dtype. */
int dmpnn_sum_act_bwd(const void* const* Z, int n_z, int64_t ldz, const void* G, int64_t ldg, const void* Ypre, int64_t ldy,
                      int dtype, int act, float act_param, void* OUT, int out_dtype, int64_t ldo, int64_t R, int64_t C,
                      void* stream);

/* Undirected averaging (base.py:202-203): OUT[r] = (f(X[r]) + f(X[rev(r)])) / 2, f = `act` on
 * load (identity for ACT_NONE).  Self-adjoint when rev is an involution, so with ACT_NONE the
 * same call is its own autograd mirror. */
int dmpnn_rev_average(const void* X, int x_dtype, int64_t ldx, const int32_t* rev_row,
                      int64_t R, int64_t C, int act, float act_param,
                      void* OUT, int out_dtype, int64_t ldo, void* stream);

/* ---------------------------------------------------------------------------------------
 * Activation backward:  dZ[r,c] = G[gi(r), c] * tau'(.)  where tau' is evaluated from
 * Yact (from_preact==0: Yact holds tau(z); from_preact!=0: Yact holds z).  If ACC != NULL,
 * ACC[r,c] += dZ[r,c] (the dH_0 accumulator of the autograd mirror of base.py:135-141).
 * dZ may be NULL when only the accumulation is wanted.
 * ------------------------------------------------------------------------------------- */
int dmpnn_act_bwd(const void* G, int g_dtype, int64_t ldg, const int32_t* gidx,
                  const void* Yact, int y_dtype, int64_t ldy, int from_preact,
                  int act, float act_param,
                  void* dZ, int dz_dtype, int64_t lddz,
                  void* ACC, int acc_dtype, int64_t ldacc,
                  int64_t R, int64_t C, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused Blackwell depth step (bf16 hidden states, tcgen05 + TMEM + TMA):
 *   H_next[rev(e')] = tau( H_0[rev(e')] + bias + W_h . ( sum_{in(v)} g(H_prev) - g(H_prev[e']) ) )
 * i.e. message (mixins.py:11-18) + update (base.py:135-141) in ONE launch, one CTA per SM,
 * molecule-aligned 128-row tiles from dmpnn_layout_build.  g = tau when first_step!=0
 * (H_prev = H_0 and H^0 = tau(H_0) is recomputed on load), identity otherwise.
 * Wpk is W_h packed by dmpnn_pack_weight_bf16.  Requires ld % 16 == 0, a 32-byte aligned H_next, h <= 304, all tiles
 * <= 128 rows, DMPNN_FLAG_REV_INVOLUTION.  Returns <0 (and does nothing) otherwise.
 * M_out (nullable; first_step only; bf16, same ld, 32-byte aligned, ld % 16 == 0): also stores the message
 * M^1[e] (mixins.py:11-18) that the step consumed, saved for the W_h gradient instead of being recomputed.
 * ------------------------------------------------------------------------------------- */
/* ---------------------------------------------------------------------------------------
 * Tensor-core linear layers of the bf16 tier (tcgen05 / TMEM / TMA), for the GEMMs outside the fused
 * depth step: W_i (mixins.py:8-9, 22-23), W_o (base.py:180-182) and dX = dY.W of their autograd mirror.
 *   dmpnn_concat_bf16     A[r] = bf16([X1[i1(r)] || X2[i2(r)] || 0..])  (torch.cat of mixins.py:9 / base.py:180)
 *   dmpnn_pack_weight_tc  nn.Linear weight (or its transpose: transpose != 0 packs B[n][k] = W[k][n]) ->
 *                         per-k-slab shared-memory images
 *   dmpnn_linear_tc_bf16  C[r, 0:N] = act(A[r, 0:K] . B^T + bias + res[r, 0:N]); A, C, res (nullable; the H_0
 *                         residual of base.py:138, ldres % 8 == 0) bf16 row-major, lda/ldc % 8 == 0,
 *                         ldc >= pad16(N), K <= 448, N <= 304; C columns [N, pad16(N)) are written as zeros.
 * ------------------------------------------------------------------------------------- */
int dmpnn_concat_bf16(const void* X1, int x1_dtype, int64_t ld1, const int32_t* idx1, int64_t K1,
                      const void* X2, int x2_dtype, int64_t ld2, const int32_t* idx2, int64_t K2,
                      void* OUT, int64_t ldo, int64_t width, int64_t R, void* stream);
/* the same gather-concatenate with an f32 result: the operands of the fp32 tier's tensor-core GEMMs (dmpnn_linear_x3) */
int dmpnn_concat_f32(const void* X1, int x1_dtype, int64_t ld1, const int32_t* idx1, int64_t K1,
                     const void* X2, int x2_dtype, int64_t ld2, const int32_t* idx2, int64_t K2,
                     float* OUT, int64_t ldo, int64_t width, int64_t R, void* stream);
int dmpnn_pack_weight_tc_bytes(int64_t N, int64_t K, size_t* bytes);
int dmpnn_pack_weight_tc(const float* W, int64_t ldw, int64_t N, int64_t K, int transpose, void* Wpk, void* stream);
int dmpnn_linear_tc_bf16(const void* A, int64_t lda, int64_t R, int64_t K, const void* Wpk, int64_t N,
                         const float* bias, const void* res, int64_t ldres, int act, float act_param,
                         void* C, int64_t ldc, void* stream);

/* Autograd mirror of one depth step on the same fused kernel (gather-by-rev mode):
 *   dOut[e] = ( sum_{e'' : src(e'') = dst(e)} dM[e''] - dM[rev(e)] ) * tau'(Yact[e]),   dM = dZ . W_h
 * computed as ((S.P) dZ) . W_h with the row mixing done on the A operand; WpkT = dmpnn_pack_weight_bf16 of W_h^T.
 * Yact = the stored activation output H^{t-1} (tau' is evaluated from it); Yact == NULL -> no mask (dH^0).
 * y_is_preact != 0: Yact holds the PRE-activation (H_0) and tau' is evaluated from it -- the t = 1 step; then
 * add0 / add1 (nullable, bf16, same ld, 16-byte aligned, must not alias dOut) are summed into the output in f32
 * before the single rounding, so that step writes dH_0 = dZ^{T-1} + .. + dZ^1 + dH^0 * tau'(H_0) directly.
 * G_out (nullable, bf16, same ld, 32-byte aligned, ld % 16 == 0): also writes the gathered operand G = (S.P) dZ, so
 * that the W_h gradient of this step is the plain GEMM dW_h += G^T . H^{t-1} (dZ^T . M^t == ((S.P) dZ)^T . H^{t-1}).
 * Same size / layout requirements as dmpnn_bond_step_fused_bf16. */
int dmpnn_bond_step_bwd_fused_bf16(const void* dZ, const void* Yact, void* dOut, int64_t ld, int64_t n_rows_alloc,
                                   int64_t h, const void* WpkT, const int32_t* rowptr, const int32_t* rev_row,
                                   const int32_t* tile_row_ptr, const int32_t* tile_atom_ptr, int64_t n_tiles,
                                   int act, float act_param, int y_is_preact, const void* add0, const void* add1,
                                   void* G_out, const int8_t* work_flag, const int32_t* n_work_dev, const int32_t* dst_row,
                                   void* stream);

/* Molecule-aligned tiles with caller-given limits (the packing rule of dmpnn_layout_build: greedy, restarted every 1024
 * molecules): tile_row_ptr / tile_atom_ptr [<= B + 1] receive the first edge row / first atom of every tile plus the end
 * sentinel, info[0..2] = tile count, max rows (edges) and max atoms of a tile.  Used for the ATOM tiles (<= 128 atoms) of
 * dmpnn_atom_step_fused_bf16.  Workspace from dmpnn_tiles_workspace_bytes; stream-ordered, no host sync. */
int dmpnn_tiles_workspace_bytes(int64_t B, size_t* bytes);
int dmpnn_tiles_build(const int32_t* mol_atom_ptr, const int32_t* mol_row_ptr, int64_t B, int row_limit, int atom_limit,
                      int32_t* tile_row_ptr, int32_t* tile_atom_ptr, int32_t* info, void* workspace, void* stream);

/* Atom-granular fused depth step -- AtomMessagePassing (chemprop/nn/message_passing/mixins.py:25-30 + base.py:135-141)
 * restated on atoms (the reference's edge state H[e] depends only on src(e)):
 *   H_next[v] = act( H_0[v] + bias + W . sum_{e in in(v)} g(H_prev[src(e)]) ),   g = act on the first step, identity after,
 * one launch: neighbour gather from the TMA-loaded atom tile + tcgen05 GEMM + epilogue, the kernel of
 * dmpnn_bond_step_fused_bf16 with its ATOM gather.  The loop-invariant bond term W_h[:, h:] . sum_in E of the reference's
 * update is folded into H_0 by the caller (engine.atom_forward_fused).  rowptr: dst-sorted CSR over atoms; nbr_row: source
 * atom of every edge row; tile_atom_ptr / tile_edge_ptr: first atom / first edge row of every atom tile (dmpnn_tiles_build
 * with atom_limit = 128) and *n_tiles_dev tiles (device scalar; n_tiles_max only sizes the checks).  Every molecule must
 * have <= 128 atoms.  N_out (first step only): the gathered operand, for the W_h gradient.  The mirror:
 *   dOut[v] = ( (sum_{e in in(v)} dZ[src(e)]) . W ) * act'(Yact[v])      (the adjacency is symmetric)
 * with the modes of dmpnn_bond_step_bwd_fused_bf16 (Yact null: no mask; y_is_preact + addends: the last step). */
int dmpnn_atom_step_fused_bf16(const void* H_prev, const void* H_0, void* H_next, int64_t ld, int64_t n_rows_alloc, int64_t h,
                               const void* Wpk, const float* bias, const int32_t* rowptr, const int32_t* nbr_row,
                               const int32_t* tile_atom_ptr, const int32_t* tile_edge_ptr, const int32_t* n_tiles_dev,
                               int64_t n_tiles_max, int act, float act_param, int first_step, void* N_out, void* stream);
int dmpnn_atom_step_bwd_fused_bf16(const void* dZ, const void* Yact, void* dOut, int64_t ld, int64_t n_rows_alloc, int64_t h,
                                   const void* WpkT, const int32_t* rowptr, const int32_t* nbr_row,
                                   const int32_t* tile_atom_ptr, const int32_t* tile_edge_ptr, const int32_t* n_tiles_dev,
                                   int64_t n_tiles_max, int act, float act_param, int y_is_preact, const void* add0,
                                   const void* add1, void* G_out, void* stream);

/* Tensor-core weight gradient (bf16 operands, f32 accumulate, deterministic two-pass reduction):
 *   dW[n, 0:K] (+)= sum_r dY[r, n] * X[r, 0:K]      dY: R x N (ld lddy), X: R x K (ld ldx), both bf16 row-major
 * N <= 384, K <= 448; lddy, ldx multiples of 8.  Workspace from dmpnn_wgrad_tc_workspace_bytes. */
int dmpnn_wgrad_tc_workspace_bytes(int64_t N, int64_t K, size_t* bytes);
int dmpnn_wgrad_tc_bf16(const void* dY, int64_t lddy, const void* X, int64_t ldx, int64_t R, int64_t N, int64_t K,
                        float* dW, int64_t lddw, int accumulate, void* workspace, void* stream);
/* The same with up to three dY terms sharing the launch:  dW (+)= sum_t dY_t^T X  (all terms R x N with one ld; X is read
 * once per stage).  2 * n_terms + ceil(K / 64) <= 9.  Used for the W_i gradient (mixins.py:8-9 under autograd), whose
 * upstream gradient dH_0 = sum_t dZ^t + dH^0 tau'(H_0) is a sum the mirror never forms. */
int dmpnn_wgrad_tc_multi_bf16(const void* const* dYs, int n_terms, int64_t lddy, const void* X, int64_t ldx, int64_t R,
                              int64_t N, int64_t K, float* dW, int64_t lddw, int accumulate, void* workspace, void* stream);
/* Column sums (bias gradient): out[n] (+)= sum_r Y[r, n].  Workspace: dmpnn_linear_wgrad_workspace_bytes(R, N, 1). */
int dmpnn_column_sum(const void* Y, int y_dtype, int64_t ldy, int64_t R, int64_t N, float* out, int accumulate,
                     void* workspace, void* stream);

/* Debug aid: when set (device pointer to n_tiles x 12 uint64, zero-filled), block 0 of the fused
 * kernel records %globaltimer stamps of its pipeline phases for its first n_tiles tiles. NULL = off. */
int dmpnn_set_trace_buffer(void* dev_ptr, int64_t n_tiles);
int dmpnn_pack_weight_bf16_bytes(int64_t N, int64_t K, size_t* bytes);
int dmpnn_pack_weight_bf16(const float* W, int64_t ldw, int64_t N, int64_t K, void* Wpk, void* stream);
int dmpnn_bond_step_fused_bf16(const void* H_prev, const void* H_0, void* H_next, int64_t ld,
                               int64_t n_rows_alloc, int64_t h,
                               const void* Wpk, const float* bias,
                               const int32_t* rowptr, const int32_t* rev_row,
                               const int32_t* tile_row_ptr, const int32_t* tile_atom_ptr, int64_t n_tiles,
                               int act, float act_param, int first_step, void* M_out,
                               const int8_t* work_flag, const int32_t* n_work_dev, const int32_t* dst_row,
                               const void* drop_bits, float drop_scale, void* stream);

/* Training-mode dropout of base.py:139 INSIDE the fused step: `drop_bits` (nullable) holds 16 keep bits per (row, 16-column
 * block) -- uint16 [n_rows][pad16(h) / 16], bit q of word j = column 16 j + q -- and the epilogue writes
 * keep ? tau(z) * drop_scale : 0 with one rounding (drop_scale = 1 / (1 - p)); no mask pass over the E x h matrix.
 * dmpnn_dropout_bits fills such an array from Philox4x32-10 (key = seed, counter = (word index, offset)): bit = [u16 >= round(p *
 * 65536)], i.e. P(drop) = p to 2^-16; the same (seed, offset) always gives the same bits. */
int dmpnn_dropout_bits(void* bits, int64_t n_rows, int64_t words_per_row, float p, uint64_t seed, uint64_t offset, void* stream);

/* Work table for batches with molecules of MORE than 128 directed edges (condensed reaction graphs, BASELINE config 4 with
 * BondMessagePassing): the layout's tiles, with every tile of > 128 rows (one oversized molecule) cut into windows of <= 128
 * consecutive rows.  Outputs: work_row_ptr / work_atom_ptr (n_work + 1 entries; capacity n_tiles + E / 128 + 2), work_flag
 * (1 = window of a cut molecule) and the device scalar n_work.  Pass work_row_ptr / work_atom_ptr as the tile tables of the
 * fused step together with work_flag, n_work and the layout's dst_row (all three NULL for batches without such molecules):
 * a flagged window gathers its sibling / reverse-edge rows from global memory instead of its shared-memory tile. */
int dmpnn_work_table_build(const int32_t* tile_row_ptr, const int32_t* tile_atom_ptr, int64_t n_tiles,
                           int32_t* work_row_ptr, int32_t* work_atom_ptr, int8_t* work_flag, int32_t* n_work, void* stream);

/* ---------------------------------------------------------------------------------------
 * fp32-ACCURATE tensor-core GEMMs of the fp32 tier (csrc/gemm_x3.cu): every product is three
 * tcgen05.mma.kind::tf32 passes over an error-free hi / lo split of both operands, f32 accumulation in TMEM --
 * the accuracy of an f32 FMA chain (the reference's ATen sgemm on base.py:135-141, 180-182) at tensor-core
 * speed; hidden size up to 4096 (BASELINE config 3: h = 600, depth 6).
 *   dmpnn_pack_weight_x3  nn.Linear weight W (N x K f32, row stride ldw; transpose != 0: B[n][k] = W[k][n]) ->
 *                         pre-split {hi, lo} shared-memory images per (128-column pass, 32-wide k slab)
 *   dmpnn_linear_x3       C[r, 0:N] = act(A[row_idx ? row_idx[r] : r, 0:K] . B^T + bias + res[r, 0:N]);  A, C, res f32
 *                         row-major; K % 4 == 0, lda / ldc / ldres % 4 == 0, 16-byte aligned bases;
 *                         C columns [N, min(ldc_pad, pad16(N))) are written as zeros.
 *   dmpnn_wgrad_x3        dW[n, 0:K] (+)= sum_r dY[r, n] * X[r, 0:K];  dY: R x N, X: R x K f32 row-major, N, K, lddy,
 *                         ldx % 4 == 0; deterministic two-pass reduction; workspace from dmpnn_wgrad_x3_workspace_bytes.
 * ------------------------------------------------------------------------------------- */
int dmpnn_pack_weight_x3_bytes(int64_t N, int64_t K, size_t* bytes);
int dmpnn_pack_weight_x3(const float* W, int64_t ldw, int64_t N, int64_t K, int transpose, void* Wpk, void* stream);
int dmpnn_linear_x3(const float* A, int64_t lda, const int32_t* row_idx, int64_t R, int64_t K, const void* Wpk,
                    int64_t N, const float* bias, const float* res, int64_t ldres, int act, float act_param,
                    float* C, int64_t ldc, int64_t ldc_pad, void* stream);
int dmpnn_wgrad_x3_workspace_bytes(int64_t N, int64_t K, size_t* bytes);
int dmpnn_wgrad_x3(const float* dY, int64_t lddy, const float* X, int64_t ldx, int64_t R, int64_t N, int64_t K,
                   float* dW, int64_t lddw, int accumulate, void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------
 * Molecule-level head of the training step (csrc/head.cu; chemprop/models/model.py:126-161):
 *   dmpnn_bn_train_fwd  nn.BatchNorm1d in training mode on X (B x d f32): Y = (X - mean) * invstd * gamma + beta with the
 *                       batch mean / biased variance; running_mean / running_var (nullable) are updated in place with
 *                       `momentum` and the unbiased variance; Xhat, save_mean, save_invstd are kept for the mirror.
 *   dmpnn_bn_bwd        dX (and dgamma, dbeta when non-null) from dY, Xhat, invstd.
 *   dmpnn_mse_loss      chemprop's MSE criterion (nn/metrics.py:78-123, 139-141): loss[0] = sum_{b,t} w[b] tw[t] m (P - Y)^2
 *                       / sum m with m = isfinite(Y) (NaN target = masked, model.py:140-141); dP (nullable) = dloss/dP.
 *   dmpnn_bce_loss      chemprop's BCELoss on logits (nn/metrics.py:292-295): P, Y are B x T; per element
 *                       L = max(z, 0) - z y + log1p(exp(-|z|)) (soft labels in [0, 1] accepted);
 *                       loss[0] = sum w[b] tw[t] m L / sum m; dP (nullable) = w tw m (sigmoid(z) - y) / sum m.
 *   dmpnn_ce_loss       chemprop's CrossEntropyLoss (nn/metrics.py:298-303): P is B x (T C), column t C + c = logit of class
 *                       c of task t (predictors.py: reshape(b, -1, C)); Y is B x T class ids; L = logsumexp(z) - z_y;
 *                       dP (nullable) = w tw m (softmax(z) - onehot(y)) / sum m.  A finite target that is not an integer
 *                       in [0, C) makes loss[0] (and that item's dP) NaN: the stand-in for torch's error, which would
 *                       need a host sync.
 *                       For both: m = isfinite(Y); loss[0] = 0 and dP = 0 when sum m = 0.  One cluster of 8 blocks
 *                       (partials combined in rank order over distributed shared memory): bit-reproducible.
 *   dmpnn_class_probs   eval output of the classification heads (predictors.py:241-244, 310-311): Q = sigmoid(P) when
 *                       C == 1, otherwise softmax over each group of C columns; P, Q are B x (T C).
 *   dmpnn_class_probs_bwd  dP = dQ q (1 - q) (C == 1) or q (dQ - <dQ, q>) per group, from the saved Q.
 * All reductions run in a fixed order (deterministic); no host synchronisation.
 * ------------------------------------------------------------------------------------- */
int dmpnn_bn_train_fwd(const float* X, int64_t ldx, int64_t B, int64_t d, const float* gamma, const float* beta,
                       float eps, float momentum, float* running_mean, float* running_var, float* Y, int64_t ldy,
                       float* Xhat, int64_t ldh, float* save_mean, float* save_invstd, void* stream);
int dmpnn_bn_bwd(const float* dY, int64_t lddy, const float* Xhat, int64_t ldh, int64_t B, int64_t d,
                 const float* gamma, const float* invstd, float* dX, int64_t lddx, float* dgamma, float* dbeta,
                 void* stream);
int dmpnn_mse_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                   const float* task_weights, int64_t B, int64_t T, float* loss, float* dP, int64_t lddp, void* stream);
int dmpnn_bce_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                   const float* task_weights, int64_t B, int64_t T, float* loss, float* dP, int64_t lddp, void* stream);
int dmpnn_ce_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                  const float* task_weights, int64_t B, int64_t T, int64_t C, float* loss, float* dP, int64_t lddp,
                  void* stream);
int dmpnn_class_probs(const float* P, int64_t ldp, int64_t B, int64_t T, int64_t C, float* Q, int64_t ldq, void* stream);
int dmpnn_class_probs_bwd(const float* Q, int64_t ldq, const float* dQ, int64_t lddq, int64_t B, int64_t T, int64_t C,
                          float* dP, int64_t lddp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DMPNN_H_ */
