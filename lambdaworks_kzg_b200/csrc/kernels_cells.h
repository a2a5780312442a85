// Host-side launch interface of the PeerDAS / EIP-7594 cell kernels (cells.cu, cells_verify.cu).  Internal; the
// public boundary is include/lwkzg.h.  SURVEY §8 f4: the reference carries the 65 G2 points this path needs but
// implements none of it (/root/reference/src/srs.rs:274, src/lib.rs:60-92).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace lw {

constexpr int N_CELLS = 128;
constexpr int CELL_ELEMS = 64;
constexpr int CELL_BYTES = 2048;
constexpr int EXT_POINTS = 8192;          // FIELD_ELEMENTS_PER_EXT_BLOB = FK20 points (64 offsets x 128 frequencies)
constexpr int CELL_NAF_BYTES = 320;       // per 128th root of unity: 160 width-4 NAF digits (int8) of each GLV half

// ---- setup
void launch_cell_twiddles(void* d_tw8192, cudaStream_t st);                       // w^k, k < 8192 (Montgomery), w = FR_ROOT_8192
void launch_cell_twiddle_naf(void* d_naf, cudaStream_t st);                       // 128 x CELL_NAF_BYTES
// pts[v * 64 + b] = s_(64 (62 - v) + b) for v <= 62, infinity above: the 64 reversed, strided, zero-padded SRS columns
void launch_cell_srs_columns(void* d_pts_xyzz, const void* d_srs_monomial_aff, cudaStream_t st);
// out[(j / 64) * 4096 + b * 64 + j % 64] = affine(pts[brp7(j) * 64 + b]): the FK20 points in MSM order
void launch_cell_fk20_points(void* d_aff_out, const void* d_pts_xyzz, cudaStream_t st);

// ---- G1 FFT of size 128 over `batch` independent vectors, one stage per launch; pts[idx * batch + item] (XYZZ).
// A warp works on ONE butterfly index for 32 items, so the (fixed) twiddle's signed-digit ladder is warp-uniform.
// dif: natural in -> bit-reversed out, butterflies (P + Q, [w](P - Q)), half = 64 .. 1
// dit: bit-reversed in -> natural out, butterflies (P + [w]Q, P - [w]Q), half = 1 .. 64
void launch_cell_g1_fft_stage(void* d_pts, int batch, int half, bool dif, bool inverse, bool upper_half_zero, const void* d_naf, cudaStream_t st);

// ---- per blob
// blob bytes -> coefficient form (Montgomery, d_coef: n x 4096 x 32 B) and, if d_cells != NULL, the 128 cells
// (n x 128 x 2048 B, field elements in the mode's byte order).  mode: 0 = coefficients big-endian reduced (reference),
// 1 = evaluations little-endian, 2 = evaluations big-endian (Deneb).  Non-canonical words are the caller's to flag
// (launch_le_blob_check); here they are reduced.
void launch_cell_poly(void* d_coef, void* d_cells, const void* d_blobs, int n, int mode, const void* d_tw8192, cudaStream_t st);
// FK20 scalars: for every offset b the circulant vector of coefficient column b, DFT_128, scaled by 1/128, canonical.
// Frequency j = 64 v + j', offset b  ->  d_scalars[((v * n + blob) * 4096 + b * 64 + j') * 8 .. +8]: each half v is a
// "blob" of 4096 scalars for the fixed-base MSM kernels, over the half's own table of the points X[v][b * 64 + j']
void launch_cell_toeplitz(void* d_scalars, const void* d_coef, int n, const void* d_tw8192, cudaStream_t st);
// Hhat[j * n + blob] = sum_b scalar(blob, j, b) * X(j, b) over the two GLV digit tables (one per half of the frequencies,
// cell_table_half_entries(c) entries each, back to back).  n >= CELL_BA_MIN_BLOBS: the batched-affine kernel in its
// segmented form, two launches; below: one warp per (blob, frequency).  d_scratch: cell_msm_scratch_bytes(n)
constexpr int CELL_BA_MIN_BLOBS = 224;
size_t cell_table_half_entries(int c);
size_t cell_msm_scratch_bytes(int n);
void launch_cell_msm(void* d_pts_xyzz, const void* d_table, int c, const void* d_scalars, int n, void* d_scratch, cudaStream_t st);
// proofs[(blob * 128 + i) * 48] = compress(pts[brp7(i) * n + blob])
void launch_cell_proofs_finalize(void* d_proofs48, const void* d_pts_xyzz, int n, cudaStream_t st);

// ---- verification / recovery (cells_verify.cu)
// cell bytes -> 64 canonical field elements each (8 u32), status 1 if a word >= r
void launch_cell_parse(void* d_evals, int* d_status, const void* d_cells, int n_cells, int mode, cudaStream_t st);
// Scalars of the two MSMs of the verification equation.  Per cell k (one warp each): the interpolation polynomial of
// its 64 evaluations over the coset h_k <w64>, weighted by r^k -> d_wcoef[k][64] (Montgomery scratch); d_rpow[k] = r^k
// (canonical).  Then d_scalars_b (canonical, 8 u32 each):
//   [0, n) r^k h_k^64 | [n, n + nc) w_i = sum of r^k over the cells of commitment i | [n + nc, n + nc + 64) minus the
//   summed interpolation coefficients
// matching the point vector proofs || commitments || g1_monomial[0..64).
void launch_cell_verify_scalars(void* d_wcoef, void* d_rpow, void* d_scalars_b, const void* d_evals, const uint64_t* d_cell_indices,
                                const uint32_t* d_commitment_indices, int n_cells, int n_commitments, const void* d_r, const void* d_tw8192, cudaStream_t st);
// r = H(domain || 4096 || 64 || n_commitments || n_cells || commitments || (commitment_index || cell_index || cell || proof)...)
void launch_cell_batch_challenge(void* d_r, const void* d_commitments48, int n_commitments, const uint32_t* d_commitment_indices, const uint64_t* d_cell_indices,
                                 const void* d_cells, const void* d_proofs48, int n_cells, int mode, cudaStream_t st);
// recovery of n_blobs blobs, one block each: n_cells (64..128) cells per blob -> coefficient form (Montgomery,
// d_coef: n_blobs x 4096 x 32 B).  Inputs are blob-major, n_blobs x n_cells: cell indices, evaluations and the per-cell
// status of launch_cell_parse.  d_status[blob] = 0, or 1 / 2 (C_KZG_BADARGS / C_KZG_ERROR: mode 0 -> 2) when an index
// is >= 128 or not strictly ascending, a word is >= r or no polynomial of degree < 4096 matches the cells; the
// coefficient row of a malformed blob is zeroed.  d_ws: n_blobs x CELL_RECOVER_WS_BYTES of workspace
constexpr size_t CELL_RECOVER_WS_BYTES = size_t(3) * EXT_POINTS * 32;
void launch_cell_recover(void* d_coef, int* d_status, void* d_ws, const void* d_evals, const int* d_cell_status, const uint64_t* d_cell_indices,
                         int n_blobs, int n_cells, int mode, const void* d_tw8192, cudaStream_t st);
// coefficient form (Montgomery) -> cells (both halves computed by FFT) -- the tail of launch_cell_poly for callers that already hold coefficients
void launch_cell_coef_to_cells(void* d_cells, const void* d_coef, int n, int mode, const void* d_tw8192, cudaStream_t st);

// ---- many independent verify_cell_kzg_proof_batch checks per launch sequence (cells_verify.cu).  A pass holds nb
// batches: batch b is the pass's cells [d_boff[b], d_boff[b + 1]); every per-cell array is indexed by the pass's cell,
// every per-batch one by the pass's batch.  Each batch owns two MSM segments over consecutive terms starting at
// cell_batch_term_base(first cell, b): n_b LHS terms r^k pi_k, then the RHS: n_b terms r^k h_k^64 pi_k, n_b commitment
// slots (w_j C_j for j < nc_b, scalar 0 above) and 64 monomial terms -s_m [tau^m]G.
__host__ __device__ inline size_t cell_batch_term_base(int first_cell, int b) { return 3 * (size_t)first_cell + 64 * (size_t)b; }
size_t cell_segmsm_terms(int n_cells, int nb);
// d_cell_status: 3 x n_cells (parse | proof decode | commitment decode).  d_bstatus[b] = 0, or 1 / 2 (C_KZG_BADARGS /
// C_KZG_ERROR: mode 0 -> 2) when a cell index is >= 128 or a status is set; commitments deduplicated per batch in order of
// first appearance: d_cidx[k] (index among the batch's distinct commitments), d_uniq[d_boff[b] + j] (first cell of
// distinct commitment j), d_nc[b]; d_cell_batch[k] = b; d_first: n_cells ints of scratch
void launch_cell_batches_prepare(int* d_bstatus, int* d_nc, uint32_t* d_cidx, uint32_t* d_uniq, int* d_first, int* d_cell_batch, const void* d_commit48,
                                 const uint64_t* d_cell_indices, const int* d_cell_status, int n_cells, const int* d_boff, int nb, int mode, cudaStream_t st);
// one warp per batch: r_b (canonical, 8 u32 each) over the batch's message as launch_cell_batch_challenge; zeros if empty
void launch_cell_batches_challenge(void* d_rs, const void* d_commit48, const uint32_t* d_uniq, const uint32_t* d_cidx, const uint64_t* d_cell_indices,
                                   const void* d_cells, const void* d_proofs48, const int* d_nc, const int* d_boff, int nb, int mode, cudaStream_t st);
// the term scalars (canonical, cell_segmsm_terms(n_cells, nb) x 8 u32); d_wcoef: n_cells x 64 x 32 B of scratch
void launch_cell_batches_scalars(void* d_wcoef, void* d_scal, const void* d_evals, const uint64_t* d_cell_indices, const uint32_t* d_cidx, const int* d_nc,
                                 const int* d_cell_batch, const int* d_boff, int n_cells, int nb, const void* d_rs, const void* d_tw8192, cudaStream_t st);
// segmented variable-base MSM: batch b's 288-byte partial (LHS at 0, 96 zero bytes, RHS at 192; big-endian affine,
// infinity as zeros); d_terms: cell_segmsm_terms(n_cells, nb) x 192 B of scratch
void launch_cell_segmsm(void* d_out288, void* d_terms, const void* d_scal, const void* d_proof_aff, const void* d_commit_aff, const void* d_mono_aff,
                        const uint32_t* d_uniq, const int* d_nc, const int* d_boff, int n_cells, int nb, cudaStream_t st);
// The per-cell inputs of a pass whose cells were generated from n_blobs blobs (cell g = 128 blob + g % 128): the blob's
// 48 commitment bytes -> d_commit48[g], its decoded commitment (affine Montgomery) -> d_commit_aff[g], cell index g % 128
// -> d_cell_indices[g], and d_commit_status[g] = d_blob_status[blob] if set (the blob's validity), else
// d_blob_status[n_blobs + blob] (the commitment's decode status).  Each commitment is decoded once per blob.
void launch_cell_blob_broadcast(void* d_commit48, void* d_commit_aff, int* d_commit_status, uint64_t* d_cell_indices, const void* d_blob_commit48,
                                const void* d_blob_aff, const int* d_blob_status, int n_blobs, cudaStream_t st);
// d_ok[b] = 0 if d_bstatus[b] != 0, 1 if batch b is empty, else d_pair_ok[b]; d_status[b] = d_bstatus[b] (d_status may be NULL)
// d_out[0, n) = value
void launch_fill_int(int* d_out, int value, int n, cudaStream_t st);
void launch_cell_batches_fold(int* d_ok, int* d_status, const int* d_pair_ok, const int* d_bstatus, const int* d_boff, int nb, cudaStream_t st);

}  // namespace lw
