/*
 * lwkzg.h -- C ABI of liblwkzg_b200.so, the B200-native (sm_100a CUDA) drop-in
 * for the EIP-4844 hot path of lambdaclass/lambdaworks_kzg.
 *
 * Part 1 is the c-kzg-4844 compatible boundary.  Every prototype and struct
 * layout is exactly what the reference exports from src/lib.rs (#[no_mangle]
 * extern "C") / declares in src/c_kzg_4844.h; the reference line each item
 * replaces is cited.  Part 2 is additive: batch / device-pointer entry points
 * (the c-kzg ABI is one blob per call) and a few utility calls used by the
 * benchmark and the tests.
 *
 * No torch / CUDA types appear in any signature: device buffers are passed as
 * plain `void *` device addresses and streams as `void *` (a cudaStream_t).
 *
 * There is NO CPU compute path behind these symbols: without a usable CUDA
 * device every compute call returns C_KZG_ERROR.
 */
#ifndef LWKZG_H
#define LWKZG_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ Part 1 */

/* reference: src/lib.rs:64-92, src/c_kzg_4844.h:38-60 */
#define BYTES_PER_COMMITMENT 48
#define BYTES_PER_PROOF 48
#define BYTES_PER_FIELD_ELEMENT 32
#define FIELD_ELEMENTS_PER_BLOB 4096
#define BYTES_PER_BLOB (FIELD_ELEMENTS_PER_BLOB * BYTES_PER_FIELD_ELEMENT)
#define TRUSTED_SETUP_NUM_G1_POINTS 4096
#define TRUSTED_SETUP_NUM_G2_POINTS 65

/* reference: src/lib.rs:94-98, src/c_kzg_4844.h:85-112 */
typedef struct { uint8_t bytes[32]; } Bytes32;
typedef struct { uint8_t bytes[48]; } Bytes48;
typedef struct { uint8_t bytes[BYTES_PER_BLOB]; } Blob;
typedef Bytes48 KZGCommitment;
typedef Bytes48 KZGProof;

/* reference: src/lib.rs:45-57, src/c_kzg_4844.h:125-130 */
typedef enum {
    C_KZG_OK = 0,  /* Success */
    C_KZG_BADARGS, /* The supplied data is invalid in some way */
    C_KZG_ERROR,   /* Internal error / any failure in MODE_REFERENCE */
    C_KZG_MALLOC,  /* Could not allocate memory */
} C_KZG_RET;

/* blst-shaped value types.  reference: src/lib.rs:100-166 (#[repr(C)]).
 * NB: the *values* stored by the reference (and by this library) are canonical
 * (non-Montgomery) integers with limbs most-significant first, affine with
 * z = 1 -- src/srs.rs:131-213 -- i.e. shape- but not value-compatible with blst. */
typedef uint64_t limb_t;
typedef struct { limb_t l[4]; } blst_fr;
typedef struct { limb_t l[6]; } blst_fp;
typedef struct { blst_fp fp[2]; } blst_fp2;
typedef struct { blst_fp x, y, z; } blst_p1;
typedef struct { blst_fp x, y; } blst_p1_affine;
typedef struct { blst_fp2 x, y, z; } blst_p2;
typedef struct { blst_fp2 x, y; } blst_p2_affine;
typedef blst_p1 g1_t;
typedef blst_p2 g2_t;
typedef blst_fr fr_t;

/* reference: src/lib.rs:173-197, src/c_kzg_4844.h:141-156 (never populated by
 * the reference: KZGSettings.fs is always NULL, src/lib.rs:754-758). */
typedef struct {
    uint64_t max_width;
    fr_t *expanded_roots_of_unity;
    fr_t *reverse_roots_of_unity;
    fr_t *roots_of_unity;
} FFTSettings;

/* reference: src/lib.rs:210-222, src/c_kzg_4844.h:161-170.
 * g1_values: 4096 x blst_p1, g2_values: 65 x blst_p2, both malloc()ed by the
 * loaders and released by free_trusted_setup.  When THIS library's loaders
 * build the struct, `fs` points at a library-owned object whose first bytes are
 * a zeroed FFTSettings followed by the device context (SRS and fixed-base
 * tables resident in HBM).  Settings assembled by hand with fs == NULL (as the
 * reference's own loaders produce) are accepted too: a device context is then
 * created on first use and cached, keyed by the pointers and a content hash. */
typedef struct {
    FFTSettings *fs;
    g1_t *g1_values;
    g2_t *g2_values;
} KZGSettings;

/* reference: src/lib.rs:709-715 (BADARGS unless n1 == 4096 && n2 == 65) */
C_KZG_RET load_trusted_setup(KZGSettings *out, const uint8_t *g1_bytes, size_t n1,
                             const uint8_t *g2_bytes, size_t n2);
/* reference: src/lib.rs:779-802 + src/srs.rs:25-128 (line-based text format: a header n1 / n2, then n1 G1 lines read
 * as MONOMIAL points, then n2 G2 lines; later lines are ignored).  This is not c-kzg-4844's trusted_setup.txt, whose
 * first G1 section is in Lagrange form: given that file, this loader reads the Lagrange points as monomial ones and,
 * in modes 1 and 2, transforms them again -- every later result is wrong and nothing reports it.  Load c-kzg files
 * with lwkzg_load_trusted_setup_file_ckzg (Part 2). */
C_KZG_RET load_trusted_setup_file(KZGSettings *out, FILE *in);
/* reference: src/lib.rs:821-829 (returns a code; c-kzg declares void) */
C_KZG_RET free_trusted_setup(KZGSettings *s);

/* reference: src/lib.rs:253-283 */
C_KZG_RET blob_to_kzg_commitment(KZGCommitment *out, const Blob *blob, const KZGSettings *s);
/* reference: src/lib.rs:300-344 */
C_KZG_RET compute_kzg_proof(KZGProof *proof_out, Bytes32 *y_out, const Blob *blob,
                            const Bytes32 *z_bytes, const KZGSettings *s);
/* reference: src/lib.rs:361-404 */
C_KZG_RET compute_blob_kzg_proof(KZGProof *out, const Blob *blob, const Bytes48 *commitment_bytes,
                                 const KZGSettings *s);
/* reference: src/lib.rs:407-453 */
C_KZG_RET verify_kzg_proof(bool *ok, const Bytes48 *commitment_bytes, const Bytes32 *z_bytes,
                           const Bytes32 *y_bytes, const Bytes48 *proof_bytes, const KZGSettings *s);
/* reference: src/lib.rs:456-505 */
C_KZG_RET verify_blob_kzg_proof(bool *ok, const Blob *blob, const Bytes48 *commitment_bytes,
                                const Bytes48 *proof_bytes, const KZGSettings *s);
/* reference: src/lib.rs:525-614 (n == 0 -> *ok = false, C_KZG_OK; n == 1 -> single path) */
C_KZG_RET verify_blob_kzg_proof_batch(bool *ok, const Blob *blobs, const Bytes48 *commitments_bytes,
                                      const Bytes48 *proofs_bytes, size_t n, const KZGSettings *s);

/* ------------------------------------------------------------------ Part 2 */
/* c-kzg-4844 (v2) trusted setups -- the Ethereum ceremony output as c-kzg ships it (trusted_setup.txt): c-kzg's
 * load_trusted_setup / load_trusted_setup_file signatures under an lwkzg_ prefix (a c-kzg binding reaches them with
 * #[link_name], INTEGRATION.md 2).
 *   Sections: 4096 G1 monomial points [tau^j]G, 4096 G1 Lagrange points [l_k(tau)]G in NATURAL order over w^k (w the
 *   4096th root of unity of the Lagrange modes), 65 G2 monomial points [tau^i]H, compressed; exactly 4096 x 48,
 *   4096 x 48 and 65 x 96 bytes.  precompute: 0..15, accepted as c-kzg accepts it; it changes no output (the FK20
 *   window is the "cell_window_bits" option).
 *   File: decimal counts 4096 and 65, then hex byte pairs -- the Lagrange points, the G2 points, the monomial points.
 *   Whitespace (spaces, LF, CRLF) may separate tokens and byte pairs, never the two digits of a pair; anything after
 *   the last point is ignored; anything else is malformed.  Arguments and the file are checked before the device is
 *   touched, so those errors are C_KZG_BADARGS without a GPU.
 *   Mode (captured at load): 0 uses the monomial section as the SRS; 1 and 2 the Lagrange section, bit-reversed, plus
 *   the monomial section for FK20 and cell verification.  g1_values, g2_values and every later output are
 *   byte-identical to load_trusted_setup on the monomial points of the same tau in the same mode, without its
 *   4096-MSM Lagrange conversion.
 *   Checks (C_KZG_BADARGS, lwkzg_last_error() names the check and the point): strict decoding as blst's (canonical x,
 *   consistent flags, on the curve, in the subgroup -- G2 included; no point at infinity); M_0 is the generator; with
 *   rho = SHA-256(domain || the three sections in file order) mod r, sum_k rho^k L_k = sum_j f_j M_j where f(w^k) =
 *   rho^k; e(sum rho^i M_(i+1), Q_0) = e(sum rho^i M_i, Q_1) over i < 4095; e(M_1, Q_i) = e(M_0, Q_(i+1)) for every
 *   i < 64.  c-kzg itself only checks that the Lagrange section is not the monomial one.
 *   Other failures: NULL pointers C_KZG_BADARGS, allocation C_KZG_MALLOC, no usable device C_KZG_ERROR; *out is
 *   untouched on any failure.
 *   Parity unpinned: the section order, the natural order of the Lagrange points and the 0..15 precompute range follow
 *   c-kzg-4844 v2's sources as recalled, not re-read; the Lagrange order agrees with consensus-specs'
 *   bit_reversal_permutation(KZG_SETUP_G1_LAGRANGE) and is pinned by the tests against [l_k(tau)]G. */
C_KZG_RET lwkzg_load_trusted_setup_ckzg(KZGSettings *out, const uint8_t *g1_monomial_bytes, uint64_t num_g1_monomial_bytes,
                                        const uint8_t *g1_lagrange_bytes, uint64_t num_g1_lagrange_bytes,
                                        const uint8_t *g2_monomial_bytes, uint64_t num_g2_monomial_bytes, uint64_t precompute);
C_KZG_RET lwkzg_load_trusted_setup_file_ckzg(KZGSettings *out, FILE *in, uint64_t precompute);

/* Additive batch API.  `status` (may be NULL) receives one C_KZG_RET per item
 * so a bad item does not poison the batch; the function's return value is
 * C_KZG_OK iff the call itself ran (per-item failures are only in `status`,
 * or -- when status == NULL -- the first failing item's code is returned).
 * Results are bit-identical to n calls of the matching Part-1 function. */

/* host buffers */
C_KZG_RET lwkzg_blob_to_kzg_commitment_batch(KZGCommitment *out, const Blob *blobs, size_t n,
                                             const KZGSettings *s, int *status);
C_KZG_RET lwkzg_compute_blob_kzg_proof_batch(KZGProof *out, const Blob *blobs,
                                             const Bytes48 *commitments, size_t n,
                                             const KZGSettings *s, int *status);
C_KZG_RET lwkzg_compute_kzg_proof_batch(KZGProof *proofs, Bytes32 *ys, const Blob *blobs,
                                        const Bytes32 *zs, size_t n, const KZGSettings *s,
                                        int *status);
/* commitment = blob_to_kzg_commitment(blob); proof = compute_blob_kzg_proof(blob, commitment) */
C_KZG_RET lwkzg_commit_and_prove_batch(KZGCommitment *commitments, KZGProof *proofs,
                                       const Blob *blobs, size_t n, const KZGSettings *s,
                                       int *status);

/* device buffers (plain device addresses on the context's GPU, 16-byte aligned: blobs are read with 128-bit
 * loads), asynchronous on `stream` (a cudaStream_t, NULL = default stream).  The calls return as soon as the
 * work is queued, so per-item failures cannot come back through the return value: d_status (n ints on the
 * device) receives one C_KZG_RET per item; NULL means the caller does not want them.  Either way the outputs
 * of failed items are zeroed.  (Items can only fail where the host API can: an invalid commitment argument,
 * or -- MODE_CKZG_LE -- a non-canonical blob word.) */
C_KZG_RET lwkzg_commit_and_prove_batch_device(void *d_commitments, void *d_proofs,
                                              const void *d_blobs, size_t n,
                                              const KZGSettings *s, void *stream, void *d_status);
C_KZG_RET lwkzg_blob_to_kzg_commitment_batch_device(void *d_commitments, const void *d_blobs,
                                                    size_t n, const KZGSettings *s, void *stream,
                                                    void *d_status);
C_KZG_RET lwkzg_compute_blob_kzg_proof_batch_device(void *d_proofs, const void *d_blobs,
                                                    const void *d_commitments, size_t n,
                                                    const KZGSettings *s, void *stream,
                                                    void *d_status);
/* verify_blob_kzg_proof_batch (src/lib.rs:525-614) with the n blobs, commitments and proofs already in device
 * memory; synchronous, the boolean comes back to the host.  Same results and error codes as the host call. */
C_KZG_RET lwkzg_verify_blob_kzg_proof_batch_device(bool *ok, const void *d_blobs,
                                                   const void *d_commitments, const void *d_proofs,
                                                   size_t n, const KZGSettings *s);

/* n independent verify_kzg_proof checks.  ok[i] / status[i] are exactly what verify_kzg_proof returns for item i. */
/* Per item, in every mode: a commitment or proof that does not decode or is not in G1, or -- modes 1 and 2 -- a z or
 * y >= r (mode 0 reduces them mod r, as the single call does) fails the item with C_KZG_BADARGS (modes 1 and 2) or
 * C_KZG_ERROR (mode 0), and ok[i] = false.  Each verdict comes from its own pairing check, never from an aggregate
 * (the reference's internal verify_kzg_proof_batch, src/lib.rs:639-692, is an aggregate with one verdict).  Whole
 * call: n == 0 returns C_KZG_OK and writes nothing; a NULL ok or input pointer returns C_KZG_BADARGS; with
 * status == NULL the first failing item's code is returned and ok is still filled.  The host form shards its items
 * over lwkzg_set_devices.  Both forms run in passes of a fixed size, so device memory stays bounded whatever n is.
 * The device form is asynchronous on `stream`: d_ok (n ints, 1 or 0) and d_status (n ints of C_KZG_RET, may be NULL)
 * are device memory, the inputs are device addresses, 16-byte aligned.  Built for throughput: one item per thread,
 * so a single opening is faster through verify_kzg_proof. */
C_KZG_RET lwkzg_verify_kzg_proofs(bool *ok, const Bytes48 *commitments, const Bytes32 *zs, const Bytes32 *ys,
                                  const Bytes48 *proofs, size_t n, const KZGSettings *s, int *status);
C_KZG_RET lwkzg_verify_kzg_proofs_device(void *d_ok, const void *d_commitments, const void *d_zs, const void *d_ys,
                                         const void *d_proofs, size_t n, const KZGSettings *s, void *stream,
                                         void *d_status);

/* K independent verify_blob_kzg_proof_batch checks, one per transaction or sidecar set.  Batch b is blobs
 * [offsets[b], offsets[b + 1]) of the flat blobs / commitments / proofs arrays; offsets (K + 1 host integers,
 * offsets[0] == 0, non-decreasing) stays on the host in the device form too.  ok[b] / status[b] are exactly what ONE
 * verify_blob_kzg_proof_batch call over that batch alone returns, in every mode:
 *  - an empty batch: ok = false in mode 0 (src/lib.rs:538-543), true in modes 1 and 2, C_KZG_OK;
 *  - one blob: verify_blob_kzg_proof's verdict (mode 0 subtracts y g1_values[0], as the single call does);
 *  - n_b >= 2 blobs: the batch's own challenge r_b, hashed over its own tuples with n_b in the header, weights
 *    r_b^0 .. r_b^(n_b - 1), y summed against the generator;
 *  - a commitment or proof that does not decode or is not in G1, or -- modes 1 and 2 -- a blob word >= r fails its
 *    own batch only: C_KZG_BADARGS (modes 1 and 2) or C_KZG_ERROR (mode 0), and ok = false.
 * Whole call: n_batches == 0 returns C_KZG_OK and writes nothing; a NULL ok or offsets, a NULL input pointer when
 * offsets[K] > 0, offsets[0] != 0, decreasing offsets, or more than 2^24 blobs return C_KZG_BADARGS; with status ==
 * NULL the first failing batch's code is returned and ok is still filled.  The host form shards whole batches over
 * lwkzg_set_devices.  Both forms run in passes of whole batches of at most "verify_super_blobs" blobs (a larger batch
 * gets a pass of its own), so device memory is bounded by that option and the largest batch, not by K.  The device
 * form is asynchronous on `stream`: d_ok (K ints, 1 or 0) and d_status (K ints of C_KZG_RET, may be NULL) are device
 * memory, the inputs are device addresses, 16-byte aligned, read in place. */
C_KZG_RET lwkzg_verify_blob_kzg_proof_batches(bool *ok, const Blob *blobs, const Bytes48 *commitments,
                                              const Bytes48 *proofs, const uint64_t *offsets, size_t n_batches,
                                              const KZGSettings *s, int *status);
C_KZG_RET lwkzg_verify_blob_kzg_proof_batches_device(void *d_ok, const void *d_blobs, const void *d_commitments,
                                                     const void *d_proofs, const uint64_t *offsets, size_t n_batches,
                                                     const KZGSettings *s, void *stream, void *d_status);
/* test hook: r_b of every batch of the last call on these settings, 32 little-endian bytes each; zeros for batches of
 * < 2 blobs */
C_KZG_RET lwkzg_debug_blob_batch_challenges(uint8_t *out32, size_t n_batches, const KZGSettings *s);

/* Generic G1 multi-scalar multiplication (the reference's g1_lincomb,
 * src/lib.rs:241-243): out = sum scalars[i] * points[i].  points: n x 96 bytes
 * canonical big-endian affine x||y (all-zero = infinity); scalars: n x 32 bytes
 * big-endian, reduced mod r; out: 48-byte compressed. Host buffers. */
C_KZG_RET lwkzg_g1_lincomb(Bytes48 *out, const uint8_t *points_xy_be, const uint8_t *scalars_be,
                           size_t n);

/* Multi-GPU batched verification building blocks (one process per GPU; the
 * caller all-gathers the tiny outputs, e.g. with NCCL):
 *   phase 1: per local blob i -> tuple_i = compress(C_i) || z_i || y_i || compress(pi_i)
 *            (160 bytes, the exact bytes hashed by src/utils.rs:166-206); any
 *            invalid item sets status and the call returns C_KZG_ERROR.
 *   phase 2: given ALL n_total tuples (gathered in rank order) and this rank's
 *            range [first, first+n_local), writes the rank's partial sums
 *            (3 points x 96 bytes canonical affine: sum r^i pi_i,
 *            sum r^i z_i pi_i, sum r^i (C_i - y_i G)).
 *   phase 3: given all ranks' partial sums, runs the 2-pairing check. */
C_KZG_RET lwkzg_verify_batch_phase1(uint8_t *tuples160, const Blob *blobs,
                                    const Bytes48 *commitments, const Bytes48 *proofs,
                                    size_t n_local, const KZGSettings *s);
C_KZG_RET lwkzg_verify_batch_phase2(uint8_t *partial288, const uint8_t *all_tuples160,
                                    size_t n_total, size_t first, size_t n_local,
                                    const KZGSettings *s);
C_KZG_RET lwkzg_verify_batch_phase3(bool *ok, const uint8_t *partials288, size_t n_ranks,
                                    const KZGSettings *s);

/* The same phases with the exchanged data in DEVICE memory, so that the all-gathers can run on it directly
 * (ncclAllGather / torch.distributed on CUDA tensors): phase 1 writes n_local tuples to d_tuples160 (blobs,
 * commitments and proofs are host pointers, or device pointers when inputs_on_device != 0); phase 2 reads all
 * n_total tuples from d_all_tuples160 and writes 288 bytes to d_partial288; phase 3 reads n_ranks x 288 bytes.
 * Each call returns when its results are complete in memory. */
C_KZG_RET lwkzg_verify_batch_phase1_device(void *d_tuples160, const void *blobs, const void *commitments,
                                           const void *proofs, size_t n_local, int inputs_on_device,
                                           const KZGSettings *s);
C_KZG_RET lwkzg_verify_batch_phase2_device(void *d_partial288, const void *d_all_tuples160,
                                           size_t n_total, size_t first, size_t n_local,
                                           const KZGSettings *s);
C_KZG_RET lwkzg_verify_batch_phase3_device(bool *ok, const void *d_partials288, size_t n_ranks,
                                           const KZGSettings *s);

/* Multi-GPU from ONE process (SURVEY.md §8b, §8e): after lwkzg_set_devices(ids, n) every host-buffer batch call
 * -- lwkzg_blob_to_kzg_commitment_batch, lwkzg_compute_blob_kzg_proof_batch, lwkzg_compute_kzg_proof_batch,
 * lwkzg_commit_and_prove_batch, verify_blob_kzg_proof_batch -- splits its items into contiguous shards over the
 * listed CUDA devices: one host thread and one stream set per device, the SRS and its digit table replicated on
 * each (built on the first such call).  Commit / proof shards need no exchange; batched verification exchanges
 * the 160-byte tuples and 288 bytes of partial sums per device (the reference's per-blob loop, src/lib.rs:562-596,
 * and its linear combination, :639-692).  Results are byte-identical to the single-device call.  n = 0 restores
 * the default (the device the settings were loaded on).  Returns 0 on success, 1 for an unknown or repeated id. */
int lwkzg_set_devices(const int *ids, int n);
int lwkzg_get_devices(int *ids, int cap);

/* ------------------------------------------------------------------ Part 3 */
/* PeerDAS / EIP-7594 cells and cell proofs (SURVEY.md §8 f4).  The reference stops before this: it loads the 65 G2
 * points such a path needs but only ever reads two (src/srs.rs:274; constants at src/lib.rs:60-92), and it has no
 * G1 FFT.  Names, argument order and error behaviour are c-kzg-4844's eip7594 API (the header the reference's
 * src/c_kzg_4844.h:85-231 grew into); semantics are consensus-specs fulu/polynomial-commitments-sampling.md, restated
 * in oracle/py/cells.py.  The calls follow the mode of the settings: in the Lagrange modes (1, 2) a blob is the
 * evaluation form and cells 0..63 of its extension are the blob itself; in MODE_REFERENCE a blob is 4096 big-endian
 * coefficients reduced mod r (src/utils.rs:27-41) and all 128 cells are computed.  Field elements inside a Cell use
 * the mode's byte order (big-endian except in MODE_CKZG_LE).  The settings must come from load_trusted_setup[_file]
 * (the Lagrange modes keep the monomial points the loader saw); hand-built Lagrange settings get C_KZG_ERROR.
 * Parity is unpinned: the known answers of these calls (tests/golden/cell_kats.json) come from the repository's own
 * oracle, not from external c-kzg / consensus-spec vectors. */
#define FIELD_ELEMENTS_PER_EXT_BLOB (2 * FIELD_ELEMENTS_PER_BLOB)
#define FIELD_ELEMENTS_PER_CELL 64
#define BYTES_PER_CELL (FIELD_ELEMENTS_PER_CELL * BYTES_PER_FIELD_ELEMENT)
#define CELLS_PER_EXT_BLOB (FIELD_ELEMENTS_PER_EXT_BLOB / FIELD_ELEMENTS_PER_CELL)
typedef struct { uint8_t bytes[BYTES_PER_CELL]; } Cell;

/* cells: CELLS_PER_EXT_BLOB cells or NULL; proofs: CELLS_PER_EXT_BLOB proofs or NULL (not both NULL).
 * Proofs are FK20 multiproofs: 128 fixed-base MSMs of 64 points over a digit table of the 8192 transformed SRS
 * points (built on the first call; "cell_window_bits"), one inverse and one forward G1 FFT of size 128. */
C_KZG_RET compute_cells_and_kzg_proofs(Cell *cells, KZGProof *proofs, const Blob *blob, const KZGSettings *s);
/* num_cells in [64, 128], cell_indices strictly ascending and < 128; either output may be NULL */
C_KZG_RET recover_cells_and_kzg_proofs(Cell *recovered_cells, KZGProof *recovered_proofs, const uint64_t *cell_indices,
                                       const Cell *cells, size_t num_cells, const KZGSettings *s);
/* one commitment per cell (repeats allowed, deduplicated as the spec does); num_cells = 0 verifies */
C_KZG_RET verify_cell_kzg_proof_batch(bool *ok, const Bytes48 *commitments_bytes, const uint64_t *cell_indices,
                                      const Cell *cells, const Bytes48 *proofs_bytes, size_t num_cells,
                                      const KZGSettings *s);
/* additive: n blobs per call (cells: n x 128, proofs: n x 128, either may be NULL); status[n] per blob, may be NULL */
C_KZG_RET lwkzg_compute_cells_and_kzg_proofs_batch(Cell *cells, KZGProof *proofs, const Blob *blobs, size_t n,
                                                   const KZGSettings *s, int *status);
/* the same on device buffers (16-byte aligned), ordered after / before work on `stream`; outputs of failed items
 * are zeroed; d_status (n ints) may be NULL */
C_KZG_RET lwkzg_compute_cells_and_kzg_proofs_batch_device(void *d_cells, void *d_proofs, const void *d_blobs, size_t n,
                                                          const KZGSettings *s, void *stream, void *d_status);
/* additive: the producer side of an EIP-7594 blob transaction in one call -- each blob is read once and gets its
 * commitment, its 128 cell proofs and, if wanted, its 128 cells.  commitments: n x 48 bytes and proofs: n x 128 proofs,
 * both required; cells: n x 128 cells or NULL.  The bytes of every blob equal those of lwkzg_blob_to_kzg_commitment_batch
 * and lwkzg_compute_cells_and_kzg_proofs_batch on it, in all three modes.  status[n] (may be NULL) gets one code per
 * blob; a blob fails only where both of those calls fail on it -- a word >= r in modes 1 and 2, C_KZG_BADARGS (mode 0
 * has no per-blob failure) -- and all its output slots, its commitment included, are left untouched.  Whole-call
 * errors: n == 0 returns C_KZG_OK and writes nothing; a NULL blobs, commitments or proofs returns C_KZG_BADARGS;
 * settings without the monomial SRS return C_KZG_ERROR; with status == NULL the first failing blob's code is returned.
 * A pass of up to "cell_chunk_blobs" blobs copies its blobs to the device once; the commitment MSM of
 * lwkzg_blob_to_kzg_commitment_batch reads them there on a stream of its own beside the FK20 pipeline.  After
 * lwkzg_set_devices the blobs are sharded over the GPUs. */
C_KZG_RET lwkzg_commit_and_compute_cells_and_kzg_proofs_batch(KZGCommitment *commitments, Cell *cells, KZGProof *proofs,
                                                              const Blob *blobs, size_t n, const KZGSettings *s, int *status);
/* the same on device buffers (16-byte aligned), asynchronous, ordered after / before work on `stream`; outputs of
 * failed blobs are zeroed; d_cells and d_status (n ints, C_KZG_RET values) may be NULL */
C_KZG_RET lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device(void *d_commitments, void *d_cells, void *d_proofs,
                                                                     const void *d_blobs, size_t n, const KZGSettings *s,
                                                                     void *stream, void *d_status);
/* additive: recover_cells_and_kzg_proofs over n blobs, each given by num_cells (64..128) of its cells.  cell_indices
 * and cells are n x num_cells, blob-major; the indices of each blob are strictly ascending and < 128 (blobs may use
 * different index sets of the same size).  recovered_cells: n x 128 cells or NULL; recovered_proofs: n x 128 proofs or
 * NULL (not both NULL).  status[n] (may be NULL) gets the code recover_cells_and_kzg_proofs would return for that blob;
 * a failed blob's output slots are left untouched.  Bytes of good blobs are identical to n single calls.  One call
 * recovers up to "cell_chunk_blobs" blobs per pass: one block per blob for the recovery proper, then the batched FK20
 * pipeline of lwkzg_compute_cells_and_kzg_proofs_batch; after lwkzg_set_devices the blobs are sharded over the GPUs.
 * Whole-call errors: n == 0 returns C_KZG_OK and writes nothing; a NULL required pointer returns C_KZG_BADARGS;
 * num_cells outside [64, 128] returns C_KZG_BADARGS (C_KZG_ERROR in MODE_REFERENCE); with status == NULL the first
 * failing blob's code is returned.  Per-blob failures (unsorted, repeated or out-of-range indices, a cell word >= r,
 * cells that fit no polynomial of degree < 4096) are C_KZG_BADARGS in modes 1 and 2, C_KZG_ERROR in mode 0. */
C_KZG_RET lwkzg_recover_cells_and_kzg_proofs_batch(Cell *recovered_cells, KZGProof *recovered_proofs,
                                                   const uint64_t *cell_indices, const Cell *cells, size_t num_cells,
                                                   size_t n, const KZGSettings *s, int *status);
/* the same on device buffers (16-byte aligned), ordered after / before work on `stream`, asynchronous; outputs of
 * failed blobs are zeroed; d_status (n ints, C_KZG_RET values) may be NULL */
C_KZG_RET lwkzg_recover_cells_and_kzg_proofs_batch_device(void *d_cells_out, void *d_proofs_out,
                                                          const void *d_cell_indices, const void *d_cells,
                                                          size_t num_cells, size_t n, const KZGSettings *s,
                                                          void *stream, void *d_status);
/* additive: K = n_batches independent verify_cell_kzg_proof_batch checks in one call (a PeerDAS node checks each data
 * column sidecar it receives as a batch of its own).  Batch b is cells [offsets[b], offsets[b+1]) of the flat arrays
 * commitments / cell_indices / cells / proofs (one commitment per cell, as in the single call).  offsets: K + 1 host
 * integers, offsets[0] == 0, non-decreasing.  ok[b] (K bools) gets the verdict of batch b alone; status[b] (may be
 * NULL) gets the code verify_cell_kzg_proof_batch would return for batch b alone, and ok[b] is false when it is not
 * C_KZG_OK.  An empty batch verifies.  A cell index >= 128, a cell word >= r, or a proof or commitment that does not
 * decode or is not in G1 fails its own batch only: C_KZG_BADARGS in modes 1 and 2, C_KZG_ERROR in mode 0.  Each batch
 * has its own challenge r_b over its own commitments, deduplicated in order of first appearance, exactly as the
 * single call.  Whole-call errors: n_batches == 0 returns C_KZG_OK and writes nothing; a NULL required pointer,
 * offsets that do not start at 0 or decrease, or more than 2^24 cells in total return C_KZG_BADARGS; with status ==
 * NULL the first failing batch's code is returned (ok is still filled).  One call runs in passes of whole batches of
 * at most "cell_chunk_blobs" x 128 cells (a larger batch gets a pass of its own); a pass is a fixed sequence of
 * launches whatever its number of batches: one hash warp per batch, one segmented MSM over all batches, one pairing
 * block per batch.  After lwkzg_set_devices the batches are sharded over the GPUs. */
C_KZG_RET lwkzg_verify_cell_kzg_proof_batches(bool *ok, const Bytes48 *commitments, const uint64_t *cell_indices,
                                              const Cell *cells, const Bytes48 *proofs, const uint64_t *offsets,
                                              size_t n_batches, const KZGSettings *s, int *status);
/* the same with commitments, cell_indices, cells and proofs in device memory (16-byte aligned); offsets stay on the
 * host (the caller knows its batch sizes, and the host plans the passes from them without a synchronisation).
 * Asynchronous, ordered after / before work on `stream`; d_ok and d_status are n_batches ints on the device (1 / 0 and
 * C_KZG_RET values), d_status may be NULL.  Indices are validated on the device: a malformed batch gets its status and
 * d_ok = 0, its later stages run on zeroed data. */
C_KZG_RET lwkzg_verify_cell_kzg_proof_batches_device(void *d_ok, const void *d_commitments, const void *d_cell_indices,
                                                     const void *d_cells, const void *d_proofs, const uint64_t *offsets,
                                                     size_t n_batches, const KZGSettings *s, void *stream, void *d_status);
/* additive: K = n_batches checks of blob transactions as the EIP-7594 network wrapper carries them (blobs, one
 * commitment per blob, CELLS_PER_EXT_BLOB cell proofs per blob, no cells).  Batch b is blobs [offsets[b], offsets[b+1])
 * (typically one transaction); offsets: K + 1 host integers, offsets[0] == 0, non-decreasing.  commitments: one per
 * blob; cell_proofs: 128 per blob, blob-major, proof j belongs to cell j.  ok[b] / status[b] (may be NULL) are exactly
 * what a caller gets from compute_cells_and_kzg_proofs on every blob of the batch -- (false, that code) if one fails --
 * and otherwise from ONE verify_cell_kzg_proof_batch over the batch's blobs in order: blob i's commitment 128 times, cell
 * indices 0..127, its cells and its 128 proofs.  So each batch has its own challenge over its commitments
 * deduplicated in order of first appearance, an empty batch verifies, and a blob word >= r (modes 1 and 2) or a
 * commitment or proof that does not decode or is not in G1 fails its own batch only: C_KZG_BADARGS in modes 1 and 2,
 * C_KZG_ERROR in mode 0.  Whole-call errors: n_batches == 0 returns C_KZG_OK and writes nothing; a NULL required
 * pointer, offsets that do not start at 0 or decrease, or more than 2^24 cells (offsets[K] > 131072 blobs) return
 * C_KZG_BADARGS; settings without the monomial SRS return C_KZG_ERROR; with status == NULL the first failing batch's
 * code is returned (ok is still filled).  The cells are computed on the GPU and never leave it, each commitment is
 * decoded once per blob, and the rest runs as lwkzg_verify_cell_kzg_proof_batches: passes of whole batches of at most
 * "cell_chunk_blobs" blobs (a larger batch gets a pass of its own), sharded over the GPUs after lwkzg_set_devices. */
C_KZG_RET lwkzg_verify_blob_cell_kzg_proof_batches(bool *ok, const Blob *blobs, const Bytes48 *commitments,
                                                   const Bytes48 *cell_proofs, const uint64_t *offsets,
                                                   size_t n_batches, const KZGSettings *s, int *status);
/* the same with blobs, commitments and cell_proofs in device memory (16-byte aligned); offsets stay on the host.
 * Asynchronous, ordered after / before work on `stream`; d_ok and d_status are n_batches ints on the device (1 / 0 and
 * C_KZG_RET values), d_status may be NULL. */
C_KZG_RET lwkzg_verify_blob_cell_kzg_proof_batches_device(void *d_ok, const void *d_blobs, const void *d_commitments,
                                                          const void *d_cell_proofs, const uint64_t *offsets,
                                                          size_t n_batches, const KZGSettings *s, void *stream,
                                                          void *d_status);
/* Test hook: the challenge r_b of every non-empty batch that the last lwkzg_verify_cell_kzg_proof_batches[_device] or
 * lwkzg_verify_blob_cell_kzg_proof_batches[_device] call on these settings derived, 32 little-endian bytes each (as
 * lwkzg_debug_batch_challenge); zeros for empty batches.  n_batches must not exceed the last call's. */
C_KZG_RET lwkzg_debug_cell_batch_challenges(uint8_t *out32, size_t n_batches, const KZGSettings *s);
/* Test hook: intermediate values of the FK20 pipeline for one blob, so a parity test can name the stage that deviates:
 * scalars = the 8192 MSM scalars DFT_128(circulant column b)_j / 128 as 32-byte little-endian integers, at index
 * (j / 64) * 4096 + b * 64 + j % 64 (the order of the two half tables);
 * hhat48 = the 128 MSM results (compressed, natural j); h48 = after the inverse G1 FFT (compressed; position p holds
 * H_brp7(p), odd positions infinity); fk20_xy96 = the 8192 FK20 points X(j, b) in the same order, canonical little-endian x || y. */
C_KZG_RET lwkzg_debug_cell_stages(uint8_t *scalars, uint8_t *hhat48, uint8_t *h48, uint8_t *fk20_xy96, const Blob *blob,
                                  const KZGSettings *s);
/* window of the FK20 digit table in use (-1 before the first cell call) */
int lwkzg_cell_window_bits(const KZGSettings *s);

/* Synthetic blobs (SURVEY.md §8d): word i of blob k = four big-endian u64 from
 * SplitMix64 seeded with 0xB2004844 ^ (k*4096+i), byte[0] &= 0x3f.  Written
 * straight into device memory so large batches never cross PCIe. */
C_KZG_RET lwkzg_synth_blobs_device(void *d_blobs, uint64_t first_blob, size_t n, void *stream);
/* same generator on the host (tests / CPU baseline feed) */
void lwkzg_synth_blob_host(uint8_t *blob, uint64_t k);

/* Integer-pipe peak probe (the roofline denominator R_int): runs a memory-free
 * IMAD micro-kernel with DISTINCT operand registers per MAC on the current
 * device and returns MAC32/s (32x32+64 multiply-accumulates per second).
 * variant 0 = carry chain of mad.lo.cc/madc.hi.cc pairs (IMAD.WIDE.U32.X, one
 * row of the Montgomery product), 1 = carry-less 64-bit columns (IMAD.WIDE.U32). */
double lwkzg_imad_peak(int variant);

/* Measurement hook for the roofline: launches the dominant kernel (the batched
 * fixed-base MSM gather over n device-resident blobs) alone, `iters` times
 * after one warm-up, bracketed by CUDA events on its own stream; returns the
 * average milliseconds per launch (< 0 on error).  blocks_per_blob 0 = auto. */
double lwkzg_bench_msm_kernel(const void *d_blobs, size_t n, int blocks_per_blob, int iters,
                              const KZGSettings *s);
/* Measurement hook for the variable-base MSM sweep (BASELINE config 5): n
 * synthetic points (pseudo-random entries of the fixed-base table, entry number
 * (t * 2654435761) mod (number of table entries) for point t) times n synthetic
 * scalars (the blob-word generator with blob id `seed`), generated on the
 * device; returns the average milliseconds per MSM (< 0 on error) and writes
 * the compressed result. */
double lwkzg_bench_var_msm(Bytes48 *out, size_t n, int iters, uint64_t seed, const KZGSettings *s);
/* Measurement hook: the last stage of a batched verification alone -- fold of the partial sums and the
 * 2-pairing check -- on what the previous verify_blob_kzg_proof_batch on these settings left in the workspace;
 * average milliseconds per run (< 0 on error). */
double lwkzg_bench_pairing(int iters, const KZGSettings *s);
/* fixed-base window actually in use for these settings (may be smaller than
 * the "window_bits" option if HBM was short), -1 on error */
int lwkzg_window_bits(const KZGSettings *s);

/* Test hook (host only, no GPU needed): the parallel byte copy that stages pageable caller buffers into the pinned
 * ring (a pool of host threads, LWKZG_STAGE_THREADS; copies below 1 MiB are a plain memcpy). */
void lwkzg_debug_stage_copy(void *dst, const void *src, size_t bytes);
/* how these settings hold their digit table: 0 = private copy, 1 = built here and published ("share_table"),
 * 2 = attached to the table another PROCESS built (CUDA IPC), 3 = shared with another settings object of this
 * process; -1 on error */
int lwkzg_table_share(const KZGSettings *s);
/* phase times of this thread's last load_trusted_setup[_file] / lwkzg_load_trusted_setup[_file]_ckzg, milliseconds
 * (0 for a phase that did not run): decoding (CUDA events: copies + decode kernels), the c-kzg setup check (CUDA
 * events: its kernels), the Lagrange conversion of the monomial loaders in modes 1 and 2 and the context build
 * (digit table included; host clock, both end in a device synchronisation).  Returns 0. */
int lwkzg_last_load_times(double *decode_ms, double *check_ms, double *convert_ms, double *build_ms);

/* Options: "window_bits" (fixed-base table window c, 4..16; default 16 = 100 GiB, the fastest; shrunk
 * automatically to what free device memory allows -- lwkzg_window_bits() tells; must
 * be set before the settings are first used), "msm_blocks_per_blob" (0 = auto),
 * "chunk_blobs" (host-batch pipeline chunk, default 256; 4 chunks in flight),
 * "msm_algo" (1 = default: batches of at least "msm_ba_min_blobs" (5) blobs use
 * the batched-affine MSM kernel, smaller ones the XYZZ kernel; 0 = XYZZ only;
 * both give identical bytes), "msm_ba_variant" (tuning: accumulators per thread
 * x threads per blob, see csrc/msm.cu), "verify_super_blobs" (blobs of a batched
 * verification staged on the device at a time, default 16384 = 2 GiB), "mode": 0 =
 * MODE_REFERENCE (default: exactly what lambdaworks_kzg computes -- big-endian
 * scalars reduced mod r, blob = monomial coefficients, every failure
 * C_KZG_ERROR), 1 = MODE_CKZG_LE (the little-endian-era c-kzg-4844 semantics of
 * the YAML vectors under the reference's tests/: canonical little-endian
 * scalars, blob = evaluations, Lagrange SRS derived at load, BADARGS for invalid
 * input, empty batch verifies), 2 = MODE_DENEB (the final EIP-4844 / mainnet wire format, the combination
 * the reference stopped short of -- it parses big-endian scalars, src/utils.rs:27-41, but left the Lagrange
 * conversion of the SRS as a TODO, src/lib.rs:760-770: big-endian CANONICAL scalars (>= r is BADARGS), blob =
 * evaluations over the bit-reversed roots of unity, Lagrange SRS derived at load, barycentric evaluation and
 * evaluation-form quotient, Fiat-Shamir of consensus-specs deneb/polynomial-commitments.md: domain ||
 * be128(4096) || blob || commitment, batch challenge domain || be64(4096) || be64(n) || tuples, digests read
 * big-endian).  The mode is captured when a KZGSettings is
 * loaded / first used.  Env: LWKZG_WINDOW_BITS, LWKZG_CHUNK_BLOBS, LWKZG_MODE,
 * LWKZG_MSM_ALGO, LWKZG_MSM_BA_MIN_BLOBS, LWKZG_SHARE_TABLE.  "verify_streams" (compute streams a batched verification
 * spreads its chunks over, default 6).  "share_table" (default 0; SURVEY 8 f2's table cache): 1 = the
 * digit table is keyed by (SRS contents, window, device) and held ONCE per GPU -- settings objects of one process share
 * it by reference count, other processes attach to it through a CUDA IPC handle published under /dev/shm (attaching
 * takes milliseconds instead of the 3.8 s build and no further 100 GiB); the process that built it must outlive the
 * ones attached to it.  A disk cache is deliberately absent: the GPU rebuilds the table at 26 GiB/s, faster than any
 * disk delivers it.  Cells: "cell_window_bits" (window of the FK20 digit table over 8192
 * points, 4..14, default 13 = 29 GiB, shrunk to what free device memory allows), "cell_chunk_blobs" (blobs per
 * pass of a cell batch, default 888: two full waves of the MSM kernel, one of the G1 FFT stage kernel).
 * Returns 0 on success. */
int lwkzg_set_option(const char *name, long value);
long lwkzg_get_option(const char *name);

/* Test hook: the batch challenge r = H(domain || 4096 || n || tuples) mod r (utils.rs:166-206) that the last
 * verify_blob_kzg_proof_batch / lwkzg_verify_batch_phase2 on these settings derived, as 32 little-endian
 * bytes.  The monolithic hash (phase 2) and the chunk-by-chunk one (single-GPU batch) must agree. */
C_KZG_RET lwkzg_debug_batch_challenge(uint8_t *out32, const KZGSettings *s);

/* kernels launched by this library since load (the bench's gpu_launches) */
uint64_t lwkzg_kernel_launches(void);
/* human-readable description of the last error on this thread ("" if none) */
const char *lwkzg_last_error(void);
const char *lwkzg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LWKZG_H */
