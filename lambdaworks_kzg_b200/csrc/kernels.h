// Host-side launch interface of the CUDA kernels (internal; the public
// boundary is include/lwkzg.h).  Every launcher enqueues on `st` and returns;
// errors are collected with cudaGetLastError by the caller.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// Kernels that run side by side in the verification pipeline all ask for the SAME shared-memory carve-out (the
// largest, like the batched-affine MSM kernel): blocks of kernels with different carve-outs do not share an SM -- it
// drains and is reconfigured between them -- which made a blob-hash kernel next to the thread-per-point decompression
// take 13 ms instead of 2.5 (DESIGN 3.5, profiles/r02_verify_notes.md).  Function attributes are per device.
#define LW_SAME_CARVEOUT(kernel)                                                                              \
  do {                                                                                                        \
    static bool lw_done_[64] = {};                                                                            \
    int lw_dev_ = 0;                                                                                          \
    if (cudaGetDevice(&lw_dev_) == cudaSuccess && lw_dev_ >= 0 && lw_dev_ < 64 && !lw_done_[lw_dev_]) {       \
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); \
      lw_done_[lw_dev_] = true;                                                                               \
    }                                                                                                         \
  } while (0)

namespace lw {

constexpr int N_POINTS = 4096;          // FIELD_ELEMENTS_PER_BLOB
constexpr int BLOB_BYTES = 4096 * 32;
constexpr int AFFINE_BYTES = 96;        // Montgomery x||y, 2 x 12 u32
constexpr int XYZZ_BYTES = 192;

uint64_t launches();                    // kernels launched so far
void count_launch(int n = 1);

// ---- setup (table.cu)
// canonical LE limbs (x||y, 24 u32 per point; all-zero = infinity) -> Montgomery
// affine; flags[i] = 1 if the point is not on the curve (infinity counts as
// "not on curve": srs.rs:155-172), flags2[i] = 1 if not in the r-torsion.
void launch_srs_import(void* d_aff_out, const void* d_canon_in, int* d_not_on_curve, int* d_not_in_subgroup, int n, cudaStream_t st);
// bases[j][i] = 2^(c j) P_i  (affine, Montgomery), j < nwin
void launch_table_bases(void* d_bases, const void* d_aff, int c, int nwin, int npoints, cudaStream_t st);
// GLV digit table (csrc/recode.cuh): entry(j, i, d) = ((j*npoints) << (c-1)) + i*cnt_j + (d-1) = d * bases[j][i],
// cnt_j = 2^(c-1) for j < nwin-1, cnt_top for the (unsigned) top window
void launch_table_fill(void* d_table, const void* d_bases, int c, int nwin, int npoints, uint32_t cnt_top, cudaStream_t st);
// window geometry of the table for 128-bit scalar halves (host mirror of csrc/recode.cuh)
int table_num_windows(int c);
uint32_t table_top_count(int c);
unsigned long long table_entries(int c, int npoints);

// ---- fixed-base MSM (msm.cu)
// scalars: n blobs of 4096 x 32 bytes; be_input: raw big-endian blob words
// (reduced mod r on the fly) or canonical little-endian u32 limbs.
// partials: n * blocks_per_blob XYZZ accumulators.
void launch_msm_gather(void* d_partials, const void* d_table, int c, const void* d_scalars, bool be_input,
                       int n_blobs, int blocks_per_blob, cudaStream_t st);
// batched-affine variant: `split` blocks per blob (1 for large batches; 2, 4, 8 when the batch alone would not fill the
// GPU: each block takes 1 / split of every thread's points), n_blobs * split XYZZ partials, plus a scratch area for the
// per-thread affine accumulators (msm_ba_scratch_bytes(n_blobs * split))
void launch_msm_gather_ba(void* d_partials, const void* d_table, int c, const void* d_scalars, bool be_input,
                          int n_blobs, void* d_scratch, cudaStream_t st, int split = 1);
size_t msm_ba_scratch_bytes(int n_blobs);
int msm_ba_threads();
int msm_ba_slots();
int msm_ba_num_variants();
int msm_ba_variant();
void msm_ba_set_variant(int v);   // tuning: index into BA_VARIANTS (accumulators per thread x threads per blob), msm.cu
// sum partials, normalise, compress.  d_aff_out (may be NULL): Montgomery affine.
void launch_msm_finalize(void* d_out48, void* d_aff_out, const void* d_partials, int parts_per_blob, int n_blobs, cudaStream_t st);
int msm_threads_per_block();

// ---- Fiat-Shamir + polynomial (poly.cu)
// SHA-256 midstate over domain || le64(4096) || le64(0) || blob[0 .. 131040)
// be_header: the 16 bytes after the domain are be128(4096) (MODE_DENEB) instead of le64(4096) || le64(0)
void launch_challenge_midstate(void* d_states, const void* d_blobs, int n, cudaStream_t st, bool latency = false, bool be_header = false);
// finish with blob tail + 48 commitment bytes -> z canonical (8 u32 LE per blob)
void launch_challenge_finish(void* d_z, const void* d_states, const void* d_blobs, const void* d_commit48, int n, cudaStream_t st, bool le_digest = false);
// z from caller bytes (big-endian, reduced)
void launch_fr_from_be(void* d_z, const void* d_z_be32, int n, cudaStream_t st);
// y = p(z), q = (p - y)/(X - z): warp per blob.  d_q (n x 4096 x 8 u32 canonical,
// may be NULL), d_y_be32 (n x 32 bytes big-endian, may be NULL), d_y (canonical u32, may be NULL)
void launch_poly_eval_quot(void* d_q, void* d_y, void* d_y_be32, const void* d_blobs, const void* d_z, int n, cudaStream_t st);

// ---- point codecs (codec.cu)
// status[i] = 0 ok / 2 (C_KZG_ERROR) rejected.  d_aff (Montgomery, may be NULL),
// d_recompressed48 (canonical re-encoding, may be NULL)
void launch_g1_decompress(void* d_aff, void* d_recompressed48, int* d_status, const void* d_in48, int n, cudaStream_t st, bool strict = false,
                          bool check_subgroup = true);
// the r-torsion test of points decoded with check_subgroup = false (d_aff must not be NULL there): status 0 / 2 (1 if strict)
void launch_g1_subgroup_check(int* d_status, const void* d_aff, int n, cudaStream_t st, bool strict = false);
void launch_status_or(int* d_status, const int* d_other, int n, cudaStream_t st);
void launch_zero_failed(void* d_out, int bytes_per_item, const int* d_status, int n, cudaStream_t st);

// ---- synthetic data + probes (misc.cu)
void launch_synth_blobs(void* d_blobs, uint64_t first_blob, size_t n, cudaStream_t st);
double run_imad_peak(int variant);

// ---- verification (verify.cu)
struct G2PreparedDev;  // opaque: line coefficients of one G2 point
size_t g2_prepared_bytes();
// canonical LE limbs x.c0,x.c1,y.c0,y.c1 (48 u32) -> prepared lines; flag = 1 if not on the twist.  n points, one block each
void launch_g2_prepare(void* d_prepared, int* d_bad, const void* d_canon_in, cudaStream_t st, int n = 1);
// bad[i] = 1 if g2 value i (canonical limbs, 48 u32 each) is not on the twist
void launch_g2_check(int* d_bad, const void* d_canon_in, int n, cudaStream_t st);
// single verification: C - y*g1_0 + z*pi  vs  pi  (SURVEY App. A.7, bilinear rearrangement)
// inputs: affine Montgomery C, pi; canonical z, y.  ok written as int.
void launch_verify_single(int* d_ok, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y,
                          const void* d_g1_0_aff, const void* d_prep0, const void* d_prep1, bool g1_0_in_subgroup, cudaStream_t st,
                          int* d_status = nullptr, int sub_code = 0);   // sub_code != 0: also run the r-torsion tests of C and pi, failure -> *d_status
// tuples: compress(C)||z||y||compress(pi) (160 B each)
void launch_make_tuples(void* d_tuples160, const void* d_c48, const void* d_z, const void* d_y, const void* d_pi48, int n, cudaStream_t st, bool le = false);
// r = H(domain || le64(4096) || le64(n_total) || tuples) -> canonical r (8 u32).  wire: 0 = reference (little-endian
// header, digest read big-endian), 1 = MODE_CKZG_LE (digest read little-endian), 2 = MODE_DENEB (be64 header fields,
// digest read big-endian)
void launch_batch_challenge(void* d_r, const void* d_tuples160, size_t n_total, cudaStream_t st, int wire = 0);
// the same hash over a block range of the message, state carried in d_state (first: start from the IV; last: absorb
// the rest of the message from blk0 on and write r).  blocks_ready(k) = full 64-byte blocks covered by the head and k tuples
size_t batch_challenge_state_bytes();
int batch_challenge_blocks_ready(size_t tuples_ready);
void launch_batch_challenge_part(void* d_r, void* d_state, const void* d_tuples160, size_t n_total, int blk0, int blk1, bool first, bool last,
                                 cudaStream_t st, int wire = 0);
// partial sums over [first, first+n_local) as two bucket MSMs (varmsm.cu): 3 affine points, canonical BE 96 B each --
// sum r^i pi_i | infinity | sum r^i z_i pi_i + sum r^i C_i - (sum r^i y_i) G.  The smaller MSM runs on st2 between
// ev_fork and ev_join; everything is ordered after earlier work on st and finished for later work on st.
void launch_batch_partials(void* d_partial288, const void* d_r, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y,
                           size_t first, int n_local, void* d_scratch, cudaStream_t st, cudaStream_t st2, cudaEvent_t ev_fork, cudaEvent_t ev_join);
size_t batch_partials_scratch_bytes(int n_local);
// sum n_ranks partial triples, then e(rhs, g2_0) * e(-proof_lincomb, g2_1) == 1
void launch_batch_final(int* d_ok, const void* d_partials288, int n_ranks, const void* d_prep0, const void* d_prep1, cudaStream_t st);
// n_checks independent checks, one block each: d_ok[i] from the 288 bytes at d_partials288 + 288 i
void launch_batch_final_each(int* d_ok, const void* d_partials288, int n_checks, const void* d_prep0, const void* d_prep1, cudaStream_t st);
// the same, check i against the neighbouring prepared points d_preps[i], d_preps[i + 1] (a chain of G2 points)
void launch_batch_final_chain(int* d_ok, const void* d_partials288, int n_checks, const void* d_preps, cudaStream_t st);

// ---- many independent single-opening checks (verify_proofs.cu), one item per thread
// d_pts[2 i] = C_i - y_i G + z_i pi_i, d_pts[2 i + 1] = -pi_i (affine Montgomery) from decoded C, pi (in G1 or infinity) and
// canonical z, y; glv_g: G is in the r-torsion
void launch_verify_proofs_g1(void* d_pts, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y, const void* d_g_aff, bool glv_g, int n,
                             cudaStream_t st);
// d_ok[i] = d_status[i] == 0 && e(d_pts[2 i], g2_0) e(d_pts[2 i + 1], g2_1) == 1
void launch_verify_proofs_pairing(int* d_ok, const int* d_status, const void* d_pts, const void* d_prep0, const void* d_prep1, int n, cudaStream_t st);

// ---- many independent blob-proof batches per pass (verify_batches.cu); batch b is the pass's blobs [d_boff[b], d_boff[b + 1])
// d_bstatus[b] = code if any of the batch's d_item_status is non-zero, else 0
void launch_blob_batches_status(int* d_bstatus, const int* d_item_status, const int* d_boff, int nb, int code, cudaStream_t st);
// r_b over the batch's tuples (160 B per blob, n_b in the header, wire as in launch_batch_challenge), zeros when n_b < 2
void launch_blob_batches_challenge(void* d_rs, const void* d_tuples160, const int* d_boff, int nb, int wire, cudaStream_t st);
// the 288-byte partial of every non-empty batch b at d_out288 + 288 d_slot[b] (d_slot[b] = -1: empty): sum r_b^j pi_j |
// infinity | sum r_b^j (C_j + z_j pi_j) - (sum r_b^j y_j) G, G = d_g_one for a one-blob batch (one_glv: it is in G1),
// else the generator.  d_scalars / d_terms: blob_batches_terms(n_items, nb) x 32 / 192 bytes of scratch
size_t blob_batches_terms(int n_items, int nb);
void launch_blob_batches_msm(void* d_out288, void* d_terms, void* d_scalars, const void* d_rs, const void* d_z, const void* d_y, const void* d_c_aff,
                             const void* d_pi_aff, const void* d_g_one, bool one_glv, const int* d_boff, const int* d_slot, int n_items, int nb,
                             cudaStream_t st);
// d_ok[b] = d_bstatus[b] ? 0 : empty batch ? empty_ok : d_pair_ok[d_slot[b]]; d_status (may be NULL) = d_bstatus
void launch_blob_batches_fold(int* d_ok, int* d_status, const int* d_pair_ok, const int* d_bstatus, const int* d_slot, int nb, bool empty_ok, cudaStream_t st);

// ---- MODE_CKZG_LE (le.cu)
void launch_write_generator(void* d_out, cudaStream_t st);                 // the G1 generator, affine Montgomery
void launch_le_roots(void* d_roots, cudaStream_t st);                      // 4096 Fr (Montgomery), bit-reversed order
void launch_le_idft_rows(void* d_rows, cudaStream_t st);                   // 4096 x 4096 canonical scalars (512 MiB)
void launch_affine_to_canon(void* d_out24, const void* d_aff, int n, cudaStream_t st);
// be = false: little-endian field elements (MODE_CKZG_LE); be = true: big-endian (MODE_DENEB, the mainnet wire format)
void launch_le_blob_check(int* d_status, const void* d_blobs, int n, cudaStream_t st, bool be = false);   // status 1 if a word >= r
void launch_le_fr_parse(void* d_out, int* d_status, const void* d_in32, int n, cudaStream_t st, bool be = false);
void launch_le_eval_quot(void* d_q, void* d_y, void* d_y_le32, const void* d_blobs, const void* d_z, const void* d_roots, int n, cudaStream_t st,
                         bool be = false);

// ---- generic (variable-base) MSM for lwkzg_g1_lincomb (varmsm.cu)
// points_in_g1: the caller vouches that every point is in the r-torsion (enables the GLV split for n <= 2^18)
void launch_var_msm(void* d_out48, const void* d_points_xy_be, const void* d_scalars_be, size_t n, void* d_scratch, cudaStream_t st,
                    bool points_in_g1 = false);
// the same pipeline on device-format inputs: Montgomery affine points known to be in G1, canonical 8 x u32 scalars;
// writes canonical big-endian affine x || y (96 bytes, all-zero = infinity)
void launch_var_msm_mont(void* d_out_affine_be96, const void* d_points_mont, const void* d_scalars_canon8, size_t n, void* d_scratch, cudaStream_t st);
size_t var_msm_scratch_bytes(size_t n);
size_t var_msm_bad_flag_offset(size_t n, bool points_in_g1 = false);
int var_msm_window_bits(size_t n);
void launch_var_msm_synth(void* d_pts_be, void* d_sc_be, const void* d_table, unsigned long long n_entries, unsigned long long seed, size_t n,
                          cudaStream_t st);  // int flag inside the scratch: 1 = some point was not on the curve

}  // namespace lw
