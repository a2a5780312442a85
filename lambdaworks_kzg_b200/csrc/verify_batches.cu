// Many independent verify_blob_kzg_proof_batch checks per call (lwkzg_verify_blob_kzg_proof_batches).  A pass holds nb
// batches; batch b is the pass's blobs [boff[b], boff[b + 1]).  Every per-blob array is indexed by the pass-local blob,
// every per-batch array by the pass-local batch.  The per-blob stages (decode, blob hash, evaluation, tuples) are the
// existing n-item kernels; the kernels here are the per-batch part, each launched once per pass whatever nb is:
//   status fold -> challenge r_b (one warp per batch) -> scalars -> segmented MSM (terms, reduce) -> pairings -> verdicts.
// Batch b checks  e(sum_j r_b^j (C_j - y_j G + z_j pi_j), g2_0) == e(sum_j r_b^j pi_j, g2_1)  (lib.rs:639-692): a batch
// of n >= 2 blobs hashes its own tuples with n in the header; a batch of one blob has the single weight 1 and subtracts
// y g1_values[0] in MODE_REFERENCE, as verify_blob_kzg_proof does (batches of two or more use the generator).
#include "batch_challenge.cuh"
#include "g1.cuh"
#include "kernels.h"

namespace lw {

constexpr int BB_THREADS = 128;

// One block per batch: bstatus[b] = code when any of the batch's blobs failed (decode, G1 membership, blob words).
__global__ void __launch_bounds__(BB_THREADS) blob_batches_status_kernel(int* __restrict__ bstatus, const int* __restrict__ item_status,
                                                                         const int* __restrict__ boff, int code) {
  const int b = blockIdx.x, e = boff[b + 1];
  bool fail = false;
  for (int i = boff[b] + threadIdx.x; i < e; i += BB_THREADS) fail = fail || item_status[i] != 0;
  fail = __syncthreads_or(fail);
  if (threadIdx.x == 0) bstatus[b] = fail ? code : 0;
}

// One warp per batch: r_b over the batch's own tuples, zeros for a batch of fewer than two blobs.
__global__ void __launch_bounds__(32) blob_batches_challenge_kernel(uint32_t* __restrict__ rs, const uint8_t* __restrict__ tuples, const int* __restrict__ boff,
                                                                    int wire_flags) {
  __shared__ uint32_t wk[64 * 32];
  __shared__ uint8_t head[32];
  const int b = blockIdx.x, s0 = boff[b], n = boff[b + 1] - s0;
  if (n < 2) {
    if (threadIdx.x < 8) rs[(size_t)b * 8 + threadIdx.x] = 0;
    return;
  }
  batch_challenge_warp(rs + (size_t)b * 8, nullptr, tuples + (size_t)s0 * 160, (unsigned long long)n, 0, 0, BCH_INIT | BCH_FINAL | wire_flags, wk, head);
}

// Term layout of a pass of n_items blobs and nb batches: blob i has terms 3i (pi_i, left side), 3i + 1 (pi_i, right
// side) and 3i + 2 (C_i, right side); batch b has term 3 n_items + b (the G term, right side).
__device__ __forceinline__ Fr fr_pow_small(const Fr& base_mont, unsigned e) {   // Montgomery in and out
  Fr pw = fr_one();
  bool started = false;
  for (int bit = 31; bit >= 0; bit--) {
    if (started) pw = fr_sqr(pw);
    if ((e >> bit) & 1u) { pw = fr_mul(pw, base_mont); started = true; }
  }
  return pw;
}

// One block per batch: scalars r^j, r^j z_i, r^j for blob i = boff[b] + j, and -sum_j r^j y_i for the G term
// (rlc_scalars_kernel's arithmetic with the weights restarting at r^0 in every batch).  Canonical scalars out.
__global__ void __launch_bounds__(BB_THREADS) blob_batches_scalars_kernel(uint32_t* __restrict__ sc, const uint32_t* __restrict__ rs, const uint32_t* __restrict__ z,
                                                                          const uint32_t* __restrict__ y, const int* __restrict__ boff, int n_items) {
  __shared__ uint32_t ysum[BB_THREADS][8];
  const int b = blockIdx.x, s0 = boff[b], n = boff[b + 1] - s0, t = threadIdx.x;
  Fr rc;
  for (int k = 0; k < 8; k++) rc.l[k] = rs[(size_t)b * 8 + k];
  const Fr rm = fr_to_mont(rc);
  Fr pw = fr_pow_small(rm, (unsigned)t);   // r^j for j = t, t + BB_THREADS, ...
  const Fr step = fr_pow_small(rm, BB_THREADS);
  Fr acc = fr_zero();
  for (int j = t; j < n; j += BB_THREADS) {
    const size_t i = (size_t)s0 + j;
    Fr zc, yc;
    for (int k = 0; k < 8; k++) { zc.l[k] = z[i * 8 + k]; yc.l[k] = y[i * 8 + k]; }
    const Fr p1 = fr_from_mont(pw);
    const Fr pz = fr_mul(pw, zc);   // mont(r^j) * canonical z = canonical r^j z
    acc = fr_add(acc, fr_mul(pw, yc));
    for (int k = 0; k < 8; k++) {
      sc[(3 * i) * 8 + k] = p1.l[k];
      sc[(3 * i + 1) * 8 + k] = pz.l[k];
      sc[(3 * i + 2) * 8 + k] = p1.l[k];
    }
    pw = fr_mul(pw, step);
  }
  for (int k = 0; k < 8; k++) ysum[t][k] = acc.l[k];
  __syncthreads();
  for (int s = BB_THREADS / 2; s > 0; s >>= 1) {
    if (t < s) {
      Fr a, c;
      for (int k = 0; k < 8; k++) { a.l[k] = ysum[t][k]; c.l[k] = ysum[t + s][k]; }
      a = fr_add(a, c);
      for (int k = 0; k < 8; k++) ysum[t][k] = a.l[k];
    }
    __syncthreads();
  }
  if (t == 0) {
    Fr tot;
    for (int k = 0; k < 8; k++) tot.l[k] = ysum[0][k];
    tot = fr_neg(tot);
    for (int k = 0; k < 8; k++) sc[((size_t)3 * n_items + b) * 8 + k] = tot.l[k];
  }
}

// Segmented MSM, pass 1: one thread per term.  C and pi passed their G1 tests (a rejected point arrives as infinity),
// so they take the GLV split.  The G term of a one-blob batch is g_one (what verify_blob_kzg_proof subtracts: g1_values[0]
// in MODE_REFERENCE, which need not be in G1 -- then a plain 255-bit ladder, one_glv = 0), of a larger batch the generator.
__global__ void __launch_bounds__(BB_THREADS) blob_batches_terms_kernel(G1Xyzz* __restrict__ out, const uint32_t* __restrict__ sc, const G1Affine* __restrict__ c_aff,
                                                                        const G1Affine* __restrict__ pi_aff, const G1Affine* __restrict__ g_one, int one_glv,
                                                                        const int* __restrict__ boff, int n_items, int nb) {
  const long t = (long)blockIdx.x * BB_THREADS + threadIdx.x;
  const long n3 = 3l * n_items;
  if (t >= n3 + nb) return;
  uint32_t k8[8];
  for (int k = 0; k < 8; k++) k8[k] = sc[(size_t)t * 8 + k];
  if (t < n3) {
    const long i = t / 3;
    out[t] = g1_mul_scalar_glv(t - 3 * i == 2 ? c_aff[i] : pi_aff[i], k8);
    return;
  }
  const int b = (int)(t - n3), n = boff[b + 1] - boff[b];
  if (n == 0) out[t] = xyzz_inf();
  else if (n > 1) out[t] = g1_mul_scalar_glv(g1a_generator(), k8);
  else out[t] = one_glv ? g1_mul_scalar_glv(*g_one, k8) : g1_mul_scalar(*g_one, k8, 8);
}

// pass 2: two blocks per non-empty batch (2b: left side, 2b + 1: right side), canonical big-endian affine into the
// batch's 288-byte partial at slot[b] (slot -1: empty batch, no partial): left side at 0, 96 zero bytes, right side at
// 192, infinity as zeros -- what batch_final_kernel reads.
__global__ void __launch_bounds__(BB_THREADS) blob_batches_reduce_kernel(uint8_t* __restrict__ out288, const G1Xyzz* __restrict__ terms, const int* __restrict__ boff,
                                                                         const int* __restrict__ slot, int n_items) {
  __shared__ G1Xyzz sh[BB_THREADS];
  const int b = blockIdx.x >> 1, rhs = blockIdx.x & 1, s0 = boff[b], e = boff[b + 1], at = slot[b];
  if (at < 0) return;   // the whole block
  G1Xyzz acc = xyzz_inf();
  for (int i = s0 + threadIdx.x; i < e; i += BB_THREADS) {
    if (rhs) {
      xyzz_add_ni(acc, terms[3 * (size_t)i + 1]);
      xyzz_add_ni(acc, terms[3 * (size_t)i + 2]);
    } else {
      xyzz_add_ni(acc, terms[3 * (size_t)i]);
    }
  }
  if (rhs && threadIdx.x == 0) xyzz_add_ni(acc, terms[3 * (size_t)n_items + b]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int d = BB_THREADS / 2; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) {
      G1Xyzz a = sh[threadIdx.x];
      xyzz_add_ni(a, sh[threadIdx.x + d]);
      sh[threadIdx.x] = a;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    uint8_t* o = out288 + (size_t)at * 288 + (rhs ? 192 : 0);
    const G1Affine a = xyzz_to_affine(sh[0]);
    if (g1a_is_inf(a)) {
      for (int k = 0; k < 96; k++) o[k] = 0;
    } else {
      fp_canon_to_be48(o, fp_from_mont(a.x));
      fp_canon_to_be48(o + 48, fp_from_mont(a.y));
    }
    if (!rhs)
      for (int k = 96; k < 192; k++) o[k] = 0;
  }
}

// verdicts: a failed batch is false, an empty one the mode's empty verdict, any other its pairing check's
__global__ void blob_batches_fold_kernel(int* __restrict__ ok, int* __restrict__ status, const int* __restrict__ pair_ok, const int* __restrict__ bstatus,
                                         const int* __restrict__ slot, int nb, int empty_ok) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const int st = bstatus[b], at = slot[b];
  ok[b] = st ? 0 : (at < 0 ? empty_ok : (pair_ok[at] != 0));
  if (status) status[b] = st;
}

// ------------------------------------------------------------------ launchers
void launch_blob_batches_status(int* d_bstatus, const int* d_item_status, const int* d_boff, int nb, int code, cudaStream_t st) {
  if (nb <= 0) return;
  blob_batches_status_kernel<<<nb, BB_THREADS, 0, st>>>(d_bstatus, d_item_status, d_boff, code);
  count_launch();
}
void launch_blob_batches_challenge(void* d_rs, const void* d_tuples160, const int* d_boff, int nb, int wire, cudaStream_t st) {
  if (nb <= 0) return;
  LW_SAME_CARVEOUT(blob_batches_challenge_kernel);
  blob_batches_challenge_kernel<<<nb, 32, 0, st>>>((uint32_t*)d_rs, (const uint8_t*)d_tuples160, d_boff, bch_wire_flags(wire));
  count_launch();
}
size_t blob_batches_terms(int n_items, int nb) { return 3 * (size_t)n_items + (size_t)nb; }
void launch_blob_batches_msm(void* d_out288, void* d_terms, void* d_scalars, const void* d_rs, const void* d_z, const void* d_y, const void* d_c_aff,
                             const void* d_pi_aff, const void* d_g_one, bool one_glv, const int* d_boff, const int* d_slot, int n_items, int nb,
                             cudaStream_t st) {
  if (nb <= 0) return;
  blob_batches_scalars_kernel<<<nb, BB_THREADS, 0, st>>>((uint32_t*)d_scalars, (const uint32_t*)d_rs, (const uint32_t*)d_z, (const uint32_t*)d_y, d_boff, n_items);
  const size_t terms = blob_batches_terms(n_items, nb);
  blob_batches_terms_kernel<<<(unsigned)((terms + BB_THREADS - 1) / BB_THREADS), BB_THREADS, 0, st>>>(
      (G1Xyzz*)d_terms, (const uint32_t*)d_scalars, (const G1Affine*)d_c_aff, (const G1Affine*)d_pi_aff, (const G1Affine*)d_g_one, one_glv ? 1 : 0, d_boff,
      n_items, nb);
  blob_batches_reduce_kernel<<<2 * nb, BB_THREADS, 0, st>>>((uint8_t*)d_out288, (const G1Xyzz*)d_terms, d_boff, d_slot, n_items);
  count_launch(3);
}
void launch_blob_batches_fold(int* d_ok, int* d_status, const int* d_pair_ok, const int* d_bstatus, const int* d_slot, int nb, bool empty_ok, cudaStream_t st) {
  if (nb <= 0) return;
  blob_batches_fold_kernel<<<(nb + 127) / 128, 128, 0, st>>>(d_ok, d_status, d_pair_ok, d_bstatus, d_slot, nb, empty_ok ? 1 : 0);
  count_launch();
}

}  // namespace lw
