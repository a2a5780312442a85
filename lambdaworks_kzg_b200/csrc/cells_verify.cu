// PeerDAS / EIP-7594: batched cell-proof verification and cell recovery (SURVEY §8 f4; restated in
// oracle/py/cells.py from consensus-specs `specs/fulu/polynomial-commitments-sampling.md` -- the reference has no
// counterpart, it only carries the G2 point [tau^64]G2 this check pairs against: /root/reference/src/srs.rs:274).
//
// verify_cell_kzg_proof_batch (the spec's universal verification equation):
//     e( sum_k r^k pi_k , [tau^64]G2 )  ==  e( sum_i w_i C_i  -  [sum_k r^k I_k(tau)]G  +  sum_k r^k h_k^64 pi_k , G2 )
// with I_k the interpolation polynomial of cell k over its coset h_k <w64> and w_i the sum of r^k over the cells that
// belong to commitment i.  The three terms of the right-hand side are ONE variable-base MSM over
// proofs || commitments || g1_monomial[0..64) (varmsm.cu), the left-hand side a second one; this file prepares their
// scalars: r (one sequential SHA-256 over everything), the per-cell inverse FFTs of size 64 and the weights.
//
// recover_cells_and_kzg_proofs: the spec's recover_polynomialcoeff -- vanishing polynomial of the missing cells,
// (E * Z) on the whole domain, division on the coset 7 * <w8192> -- as one block working out of shared memory.
#include "kernels_cells.h"
#include "field.cuh"
#include "g1.cuh"
#include "kernels.h"
#include "sha256.cuh"

namespace lw {

namespace {

__device__ __forceinline__ Fr fr_const(const uint32_t* c) { Fr r; for (int i = 0; i < 8; i++) r.l[i] = c[i]; return r; }
__device__ __forceinline__ uint32_t brp7(uint32_t i) { return __brev(i) >> 25; }
__device__ __forceinline__ Fr fr_pow_small(Fr base, uint32_t e) {
  Fr acc = fr_one();
  for (int bit = 31; bit >= 0; bit--) {
    acc = fr_sqr(acc);
    if ((e >> bit) & 1u) acc = fr_mul(acc, base);
  }
  return acc;
}
template <int N>
__device__ __forceinline__ Fr sm_load(const uint32_t* sm, int i) {
  Fr r;
#pragma unroll
  for (int l = 0; l < 8; l++) r.l[l] = sm[l * N + i];
  return r;
}
template <int N>
__device__ __forceinline__ void sm_store(uint32_t* sm, int i, const Fr& v) {
#pragma unroll
  for (int l = 0; l < 8; l++) sm[l * N + i] = v.l[l];
}
// In-place FFT passes over N elements in shared memory (see cells.cu); tw = powers of w8192.
template <int N>
__device__ void sm_dit(uint32_t* sm, const Fr* __restrict__ tw, bool inverse) {   // bit-reversed in -> natural out
  for (int half = 1; half < N; half <<= 1) {
    const int step = (EXT_POINTS / 2) / half;
    for (int t = threadIdx.x; t < N / 2; t += blockDim.x) {
      const int j = t & (half - 1);
      const int i0 = ((t - j) << 1) + j, i1 = i0 + half;
      Fr u = sm_load<N>(sm, i0), v = sm_load<N>(sm, i1);
      if (j) v = fr_mul(v, tw[inverse ? ((EXT_POINTS - step * j) & (EXT_POINTS - 1)) : step * j]);
      sm_store<N>(sm, i0, fr_add(u, v));
      sm_store<N>(sm, i1, fr_sub(u, v));
    }
    __syncthreads();
  }
}
template <int N>
__device__ void sm_dif(uint32_t* sm, const Fr* __restrict__ tw, bool inverse) {   // natural in -> bit-reversed out
  for (int half = N / 2; half >= 1; half >>= 1) {
    const int step = (EXT_POINTS / 2) / half;
    for (int t = threadIdx.x; t < N / 2; t += blockDim.x) {
      const int j = t & (half - 1);
      const int i0 = ((t - j) << 1) + j, i1 = i0 + half;
      Fr u = sm_load<N>(sm, i0), v = sm_load<N>(sm, i1);
      sm_store<N>(sm, i0, fr_add(u, v));
      Fr d = fr_sub(u, v);
      if (j) d = fr_mul(d, tw[inverse ? ((EXT_POINTS - step * j) & (EXT_POINTS - 1)) : step * j]);
      sm_store<N>(sm, i1, d);
    }
    __syncthreads();
  }
}

// canonical field element from 32 wire bytes; ok = false if the value is >= r
__device__ __forceinline__ Fr fr_parse_wire(const uint8_t* p, int mode, bool& ok) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
  const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = mode == 1 ? w[i] : bswap32(w[7 - i]);
  uint32_t t[8];
  ok = limbs_sub<8>(t, r.l, k::FR_MOD) != 0;   // borrow <=> r.l < modulus
  return r;
}

__global__ void cell_parse_kernel(uint32_t* __restrict__ evals, int* __restrict__ status, const uint8_t* __restrict__ cells, int n_cells, int mode) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)n_cells * CELL_ELEMS) return;
  bool ok;
  Fr v = fr_parse_wire(cells + (size_t)t * 32, mode, ok);
  if (!ok) {
    atomicOr(&status[t / CELL_ELEMS], mode == 0 ? 2 : 1);
    v = fr_zero();
  }
  uint4* dst = reinterpret_cast<uint4*>(evals + (size_t)t * 8);
  dst[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  dst[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

// ------------------------------------------------------------------ batch challenge
// message = domain(16) || u64(4096) || u64(64) || u64(n_commitments) || u64(n_cells) || commitments ||
//           for every cell: u64(commitment index) || u64(cell index) || cell (2048) || proof (48)
// Every piece is a multiple of 4 bytes; the message is addressed in big-endian 32-bit words.
struct CellMsg {
  const uint32_t* commitments;   // 12 words each
  const uint32_t* uniq;          // NULL: commitment j is commitments[j]; else it is the commitment of cell uniq[j]
  const uint32_t* commitment_indices;
  const uint64_t* cell_indices;
  const uint32_t* cells;         // 512 words each
  const uint32_t* proofs;        // 12 words each
  uint32_t head[12];
  unsigned long long n_commitments, n_cells;
  int le;                        // little-endian integers (MODE_CKZG_LE)
  __host__ __device__ static uint32_t bswap(uint32_t v) { return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24); }
  // domain || u64(4096) || u64(64) || u64(n_commitments) || u64(n_cells), from n_commitments / n_cells / le
  __host__ __device__ void set_head() {
    const uint32_t dom[4] = {0x52434b5au, 0x47434241u, 0x5443485fu, 0x5f56315fu};   // "RCKZGCBATCH__V1_"
    for (int i = 0; i < 4; i++) head[i] = dom[i];
    const unsigned long long v[4] = {4096ull, (unsigned long long)CELL_ELEMS, n_commitments, n_cells};
    for (int i = 0; i < 4; i++) {
      if (le) { head[4 + 2 * i] = bswap((uint32_t)v[i]); head[5 + 2 * i] = bswap((uint32_t)(v[i] >> 32)); }
      else { head[4 + 2 * i] = (uint32_t)(v[i] >> 32); head[5 + 2 * i] = (uint32_t)v[i]; }
    }
  }
  __device__ __forceinline__ void u64_words(uint32_t* out2, unsigned long long v) const {
    if (le) { out2[0] = bswap32((uint32_t)v); out2[1] = bswap32((uint32_t)(v >> 32)); }
    else { out2[0] = (uint32_t)(v >> 32); out2[1] = (uint32_t)v; }
  }
  __device__ __forceinline__ unsigned long long total_words() const { return 12ull + 12ull * n_commitments + 528ull * n_cells; }
  __device__ __forceinline__ uint32_t word(unsigned long long wi) const {
    if (wi < 12) return head[wi];
    wi -= 12;
    if (wi < 12ull * n_commitments) {
      if (!uniq) return bswap32(__ldg(commitments + wi));
      return bswap32(__ldg(commitments + (size_t)__ldg(uniq + wi / 12) * 12 + wi % 12));
    }
    wi -= 12ull * n_commitments;
    const unsigned long long kk = wi / 528;
    const uint32_t o = (uint32_t)(wi % 528);
    if (o < 4) {
      uint32_t two[2];
      u64_words(two, o < 2 ? (unsigned long long)__ldg(commitment_indices + kk) : (unsigned long long)__ldg(cell_indices + kk));
      return two[o & 1];
    }
    if (o < 516) return bswap32(__ldg(cells + kk * 512 + (o - 4)));
    return bswap32(__ldg(proofs + kk * 12 + (o - 516)));
  }
};

// r = SHA-256(message) mod r (canonical limbs) by one warp; wk: 64 x 32 words of shared memory
__device__ void cell_challenge_warp(uint32_t* __restrict__ r_out, const CellMsg& msg, uint32_t* wk) {
  const int lane = threadIdx.x;
  const unsigned long long words = msg.total_words();
  const int nfull = (int)(words / 16);
  Sha256State s;
  sha256_init(s);
  sha256_warp_blocks(s, nfull, [&](int blk, uint32_t* w) {
    for (int i = 0; i < 16; i++) w[i] = msg.word(16ull * blk + i);
  }, wk);
  if (lane != 0) return;
  uint32_t tail[32];
  const int rem = (int)(words - 16ull * nfull);
  for (int i = 0; i < 32; i++) tail[i] = 0;
  for (int i = 0; i < rem; i++) tail[i] = msg.word(16ull * nfull + i);
  tail[rem] = 0x80000000u;
  const int tl = (rem + 3 <= 16) ? 16 : 32;   // 0x80 word + two length words must fit
  const unsigned long long bits = words * 32ull;
  tail[tl - 2] = (uint32_t)(bits >> 32);
  tail[tl - 1] = (uint32_t)bits;
  for (int o = 0; o < tl; o += 16) sha256_compress(s, tail + o);
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = msg.le ? bswap32(s.h[i]) : s.h[7 - i];
  mod_reduce_small<FrCfg, 2>(r.l);
  for (int i = 0; i < 8; i++) r_out[i] = r.l[i];
}

__global__ void __launch_bounds__(32) cell_batch_challenge_kernel(uint32_t* __restrict__ r_out, CellMsg msg) {
  __shared__ uint32_t wk[64 * 32];
  cell_challenge_warp(r_out, msg, wk);
}

// ------------------------------------------------------------------ scalars of the two MSMs
// One warp per cell: a = IDFT_64 of the cell's evaluations (given in bit-reversed order), coefficient m of the
// interpolation polynomial = a_m h^-m / 64; weighted by r^k and written to wcoef[k][m] (Montgomery).
// Lane 0 also writes r^k (rpow, canonical) and r^k h^64 (scalars_b[k], canonical).
// BATCHED: cell kq belongs to batch b = cell_batch[kq] with cells [boff[b], boff[b + 1]) and challenge r_canon[b]; k is
// its index inside the batch, and r^k / r^k h^64 go to terms base + k / base + n_b + k of the batch's MSM segments
// (rpow == scalars_b: the term scalars of cell_batch_term_base).
template <bool BATCHED>
__global__ void __launch_bounds__(32) cell_interp_kernel(Fr* __restrict__ wcoef, uint32_t* rpow, uint32_t* scalars_b,
                                                        const uint32_t* __restrict__ evals, const uint64_t* __restrict__ cell_indices,
                                                        const uint32_t* __restrict__ r_canon, const Fr* __restrict__ tw,
                                                        const int* __restrict__ cell_batch, const int* __restrict__ boff) {
  __shared__ uint32_t sm[8 * 64];
  const int kq = blockIdx.x, lane = threadIdx.x;
  uint32_t k = (uint32_t)kq;
  size_t ia = (size_t)kq, ib = (size_t)kq;
  if (BATCHED) {
    const int b = cell_batch[kq], s0 = boff[b], n = boff[b + 1] - s0;
    k = (uint32_t)(kq - s0);
    r_canon += (size_t)b * 8;
    ia = cell_batch_term_base(s0, b) + k;
    ib = ia + (size_t)n;
  }
  const uint32_t hexp = brp7((uint32_t)cell_indices[kq] & 127u);   // h_k = w8192^brp7(cell index)
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = r_canon[i];
  const Fr rk = fr_pow_small(fr_to_mont(r), k);
  for (int i = lane; i < 64; i += 32) {
    Fr v;
    for (int l = 0; l < 8; l++) v.l[l] = evals[((size_t)kq * 64 + i) * 8 + l];
    sm_store<64>(sm, i, fr_to_mont(v));
  }
  __syncthreads();
  sm_dit<64>(sm, tw, true);
  const Fr scale = fr_mul(rk, fr_const(k::FR_INV_64));
  for (int m = lane; m < 64; m += 32) {
    const uint32_t e = (EXT_POINTS - ((hexp * (uint32_t)m) & (EXT_POINTS - 1))) & (EXT_POINTS - 1);
    wcoef[(size_t)kq * 64 + m] = fr_mul(fr_mul(sm_load<64>(sm, m), tw[e]), scale);
  }
  if (lane == 0) {
    const Fr a = fr_from_mont(rk), b = fr_from_mont(fr_mul(rk, tw[64u * hexp]));
    for (int l = 0; l < 8; l++) { rpow[ia * 8 + l] = a.l[l]; scalars_b[ib * 8 + l] = b.l[l]; }
  }
}

// scalars_b layout: [0, n) r^k h_k^64 (proofs) | [n, n + nc) commitment weights | [n + nc, n + nc + 64) minus the summed
// interpolation coefficients (g1_monomial[0..64))
__global__ void __launch_bounds__(128) cell_verify_finish_kernel(uint32_t* __restrict__ scalars_b, const Fr* __restrict__ wcoef, const uint32_t* __restrict__ rpow,
                                                                const uint32_t* __restrict__ commitment_indices, int n, int nc) {
  const int t = threadIdx.x;
  if (t < 64) {
    Fr acc = fr_zero();
    for (int kq = 0; kq < n; kq++) acc = fr_add(acc, wcoef[(size_t)kq * 64 + t]);
    const Fr v = fr_from_mont(fr_neg(acc));
    for (int l = 0; l < 8; l++) scalars_b[((size_t)n + nc + t) * 8 + l] = v.l[l];
  }
  for (int i = t; i < nc; i += blockDim.x) {
    Fr acc = fr_zero();
    for (int kq = 0; kq < n; kq++) {
      if ((int)commitment_indices[kq] == i) {
        Fr v;
        for (int l = 0; l < 8; l++) v.l[l] = rpow[(size_t)kq * 8 + l];
        acc = fr_add(acc, v);   // canonical + canonical mod r
      }
    }
    for (int l = 0; l < 8; l++) scalars_b[((size_t)n + i) * 8 + l] = acc.l[l];
  }
}

// ------------------------------------------------------------------ many independent batches per call
// A pass holds nb batches; batch b is the pass's cells [boff[b], boff[b + 1]).  Every per-cell array is indexed by the
// pass-local cell, every per-batch array by the pass-local batch.

// One block per batch: folds the per-cell statuses (parse | proof decode | commitment decode, 3 x n_cells) and the
// index range into the batch's status, and deduplicates its commitments in order of first appearance:
// cidx[k] = index of cell k's commitment among the batch's distinct ones, uniq[boff[b] + j] = the first cell holding
// distinct commitment j, nc[b] = their number.  first: n_cells ints of scratch.
__global__ void __launch_bounds__(256) cell_batches_prepare_kernel(int* __restrict__ bstatus, int* __restrict__ nc, uint32_t* __restrict__ cidx,
                                                                  uint32_t* __restrict__ uniq, int* __restrict__ first, int* __restrict__ cell_batch,
                                                                  const uint8_t* __restrict__ commit48, const uint64_t* __restrict__ cell_indices,
                                                                  const int* __restrict__ cell_status, int n_cells, const int* __restrict__ boff, int mode) {
  __shared__ int n_uniq;
  const int b = blockIdx.x, s0 = boff[b], e = boff[b + 1];
  if (threadIdx.x == 0) n_uniq = 0;
  bool fail = false;
  for (int g = s0 + threadIdx.x; g < e; g += blockDim.x) {
    cell_batch[g] = b;
    fail = fail || cell_indices[g] >= (uint64_t)N_CELLS || cell_status[g] || cell_status[n_cells + g] || cell_status[2 * n_cells + g];
    const uint4* mine = reinterpret_cast<const uint4*>(commit48 + (size_t)g * 48);
    const uint4 m0 = mine[0], m1 = mine[1], m2 = mine[2];
    int f = g;
    for (int j = s0; j < g; j++) {
      const uint4* o = reinterpret_cast<const uint4*>(commit48 + (size_t)j * 48);
      const uint4 o0 = o[0];
      if (o0.x != m0.x || o0.y != m0.y || o0.z != m0.z || o0.w != m0.w) continue;
      const uint4 o1 = o[1], o2 = o[2];
      if (o1.x == m1.x && o1.y == m1.y && o1.z == m1.z && o1.w == m1.w && o2.x == m2.x && o2.y == m2.y && o2.z == m2.z && o2.w == m2.w) { f = j; break; }
    }
    first[g] = f;
  }
  fail = __syncthreads_or(fail);
  int mine_uniq = 0;
  for (int g = s0 + threadIdx.x; g < e; g += blockDim.x) {
    const int f = first[g];
    uint32_t cnt = 0;
    for (int j = s0; j < f; j++) cnt += first[j] == j;
    cidx[g] = cnt;
    if (f == g) { uniq[s0 + cnt] = (uint32_t)g; mine_uniq++; }
  }
  if (mine_uniq) atomicAdd(&n_uniq, mine_uniq);
  __syncthreads();
  if (threadIdx.x == 0) {
    nc[b] = n_uniq;
    bstatus[b] = fail ? (mode == 0 ? 2 : 1) : 0;   // C_KZG_ERROR in MODE_REFERENCE, C_KZG_BADARGS in the c-kzg modes
  }
}

// One warp per batch: its challenge r_b over the batch's own message (the single call's), zeros for an empty batch.
__global__ void __launch_bounds__(32) cell_batches_challenge_kernel(uint32_t* __restrict__ rs, const uint32_t* __restrict__ commit, const uint32_t* __restrict__ uniq,
                                                                   const uint32_t* __restrict__ cidx, const uint64_t* __restrict__ cell_indices,
                                                                   const uint32_t* __restrict__ cells, const uint32_t* __restrict__ proofs,
                                                                   const int* __restrict__ nc, const int* __restrict__ boff, int le) {
  __shared__ uint32_t wk[64 * 32];
  const int b = blockIdx.x, s0 = boff[b], n = boff[b + 1] - s0;
  if (n == 0) {
    if (threadIdx.x < 8) rs[(size_t)b * 8 + threadIdx.x] = 0;
    return;
  }
  CellMsg m;
  m.commitments = commit;
  m.uniq = uniq + s0;
  m.commitment_indices = cidx + s0;
  m.cell_indices = cell_indices + s0;
  m.cells = cells + (size_t)s0 * 512;
  m.proofs = proofs + (size_t)s0 * 12;
  m.n_commitments = (unsigned long long)nc[b];
  m.n_cells = (unsigned long long)n;
  m.le = le;
  m.set_head();
  cell_challenge_warp(rs + (size_t)b * 8, m, wk);
}

// One block per batch: the scalars of the monomial terms (minus the summed interpolation coefficients) and of the
// commitment slots (w_j = sum of r^k over the batch's cells with commitment j, 0 for the unused slots j >= nc).
__global__ void __launch_bounds__(128) cell_batches_finish_kernel(uint32_t* __restrict__ scal, const Fr* __restrict__ wcoef, const uint32_t* __restrict__ cidx,
                                                                 const int* __restrict__ nc, const int* __restrict__ boff) {
  const int b = blockIdx.x, s0 = boff[b], n = boff[b + 1] - s0, t = threadIdx.x;
  const size_t base = cell_batch_term_base(s0, b);
  if (t < 64) {
    Fr acc = fr_zero();
    for (int k = 0; k < n; k++) acc = fr_add(acc, wcoef[(size_t)(s0 + k) * 64 + t]);
    const Fr v = fr_from_mont(fr_neg(acc));
    for (int l = 0; l < 8; l++) scal[(base + 3 * (size_t)n + t) * 8 + l] = v.l[l];
  }
  const int nb_c = nc[b];
  for (int j = t; j < n; j += blockDim.x) {
    Fr acc = fr_zero();
    if (j < nb_c) {
      for (int k = 0; k < n; k++) {
        if ((int)cidx[s0 + k] == j) {
          Fr v;
          for (int l = 0; l < 8; l++) v.l[l] = scal[(base + k) * 8 + l];   // r^k, canonical
          acc = fr_add(acc, v);
        }
      }
    }
    for (int l = 0; l < 8; l++) scal[(base + 2 * (size_t)n + j) * 8 + l] = acc.l[l];
  }
}

// Segmented variable-base MSM, pass 1: one thread per (point, scalar) term, [s]P by the GLV split (every point passed
// the G1 check or is a monomial SRS point).  The batch of term t is found by bisection over the term bases.
__global__ void __launch_bounds__(128) cell_segmsm_terms_kernel(G1Xyzz* __restrict__ out, const uint32_t* __restrict__ scal, const G1Affine* __restrict__ proof_pts,
                                                               const G1Affine* __restrict__ commit_pts, const G1Affine* __restrict__ mono,
                                                               const uint32_t* __restrict__ uniq, const int* __restrict__ nc, const int* __restrict__ boff,
                                                               int nb, long n_terms) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_terms) return;
  int lo = 0, hi = nb - 1;   // the last batch whose base is <= t
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((long)cell_batch_term_base(boff[mid], mid) <= t) lo = mid;
    else hi = mid - 1;
  }
  const int b = lo, s0 = boff[b], n = boff[b + 1] - s0;
  const long u = t - (long)cell_batch_term_base(s0, b);
  G1Affine p;
  bool use = true;
  if (u < n) p = proof_pts[s0 + u];                       // LHS: r^k pi_k
  else if (u < 2 * n) p = proof_pts[s0 + u - n];          // RHS: r^k h_k^64 pi_k
  else if (u < 3 * n) {                                   // RHS: w_j C_j
    const int j = (int)(u - 2 * n);
    use = j < nc[b];
    p = commit_pts[use ? uniq[s0 + j] : 0];
  } else p = mono[u - 3 * n];                             // RHS: -s_m [tau^m]G
  uint32_t k8[8];
  for (int l = 0; l < 8; l++) k8[l] = scal[(size_t)t * 8 + l];
  out[t] = use ? g1_mul_scalar_glv(p, k8) : xyzz_inf();
}

// pass 2: one block per segment (2b: LHS of batch b, 2b + 1: RHS), affine big-endian into the batch's 288-byte
// partial: LHS at 0, 96 zero bytes, RHS at 192, infinity as zeros (what batch_final_kernel reads)
__global__ void __launch_bounds__(128) cell_segmsm_reduce_kernel(uint8_t* __restrict__ out288, const G1Xyzz* __restrict__ terms, const int* __restrict__ boff) {
  __shared__ G1Xyzz sh[128];
  const int b = blockIdx.x >> 1, rhs = blockIdx.x & 1, s0 = boff[b], n = boff[b + 1] - s0;
  const size_t base = cell_batch_term_base(s0, b);
  const size_t lo = rhs ? base + n : base, hi = rhs ? base + 3 * (size_t)n + 64 : base + n;
  G1Xyzz acc = xyzz_inf();
  for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) xyzz_add_ni(acc, terms[i]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int d = blockDim.x / 2; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) {
      G1Xyzz a = sh[threadIdx.x];
      xyzz_add_ni(a, sh[threadIdx.x + d]);
      sh[threadIdx.x] = a;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    uint8_t* o = out288 + (size_t)b * 288 + (rhs ? 192 : 0);
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

// Cells generated from blobs: one block of 128 threads per blob, thread k of blob b writes cell 128 b + k's inputs of
// the pass -- the blob's commitment bytes (read by the deduplication and the hash), its decoded point (the segmented
// MSM), its status (a blob word >= r, else the commitment's decode status) and the cell index k.
__global__ void __launch_bounds__(128) cell_blob_broadcast_kernel(uint8_t* __restrict__ commit48, G1Affine* __restrict__ commit_pts, int* __restrict__ commit_status,
                                                                 uint64_t* __restrict__ cell_indices, const uint8_t* __restrict__ blob_commit48,
                                                                 const G1Affine* __restrict__ blob_pts, const int* __restrict__ blob_status, int n_blobs) {
  const int b = blockIdx.x, k = threadIdx.x;
  const size_t g = (size_t)b * N_CELLS + k;
  const uint4* src = reinterpret_cast<const uint4*>(blob_commit48 + (size_t)b * 48);
  uint4* dst = reinterpret_cast<uint4*>(commit48 + g * 48);
  dst[0] = src[0];
  dst[1] = src[1];
  dst[2] = src[2];
  commit_pts[g] = blob_pts[b];
  const int valid = blob_status[b];
  commit_status[g] = valid ? valid : blob_status[n_blobs + b];
  cell_indices[g] = (uint64_t)k;
}

__global__ void fill_int_kernel(int* __restrict__ out, int v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

// verdicts: a failed batch is false, an empty one true, any other the pairing check's
__global__ void cell_batches_fold_kernel(int* __restrict__ ok, int* __restrict__ status, const int* __restrict__ pair_ok, const int* __restrict__ bstatus,
                                         const int* __restrict__ boff, int nb) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const int st = bstatus[b];
  ok[b] = st ? 0 : (boff[b + 1] == boff[b] ? 1 : (pair_ok[b] != 0));
  if (status) status[b] = st;
}

// ------------------------------------------------------------------ recovery
// One block of 512 threads per blob.  Its global scratch holds 3 x 8192 field elements; an 8192-point transform is one
// radix-2 pass through global memory plus two 4096-point transforms in shared memory.
constexpr int REC_THREADS = 512;
constexpr int REC_SMEM = 4096 * 32;

// x (natural order, 8192 in global) -> X (natural order): DIF top stage, two 4096-point DIFs, un-bit-reverse on store
__device__ void fft8192(Fr* __restrict__ out, const Fr* __restrict__ in, uint32_t* sm, const Fr* __restrict__ tw, bool inverse) {
  for (int h = 0; h < 2; h++) {
    for (int i = threadIdx.x; i < 4096; i += blockDim.x) {
      const Fr u = in[i], v = in[i + 4096];
      Fr x = h == 0 ? fr_add(u, v) : fr_mul(fr_sub(u, v), tw[inverse ? ((EXT_POINTS - i) & (EXT_POINTS - 1)) : i]);
      sm_store<4096>(sm, i, x);
    }
    __syncthreads();
    sm_dif<4096>(sm, tw, inverse);
    // position p of sub-transform h holds X[2 * brp12(p) + h]
    for (int p = threadIdx.x; p < 4096; p += blockDim.x) out[2 * (__brev((uint32_t)p) >> 20) + h] = sm_load<4096>(sm, p);
    __syncthreads();
  }
}

// Block b recovers blob b from its n_cells cells: indices, parsed evaluations and per-cell parse status at
// b * n_cells; it writes 4096 coefficients at coef_out + b * 4096 and status[b] (0, or 1 / 2 = C_KZG_BADARGS /
// C_KZG_ERROR by mode, as cell_parse_kernel).  The indices live on the device, so they are validated here: a blob
// with an index >= 128, indices not strictly ascending or a word >= r gets a zero coefficient row, so that the later
// stages of the pass read initialised memory.
__global__ void __launch_bounds__(REC_THREADS) cell_recover_kernel(Fr* __restrict__ coef_out, int* __restrict__ status, Fr* __restrict__ ws,
                                                                  const uint32_t* __restrict__ evals, const int* __restrict__ cell_status,
                                                                  const uint64_t* __restrict__ cell_indices, int n_cells, int mode,
                                                                  const Fr* __restrict__ tw) {
  extern __shared__ uint32_t sm[];
  __shared__ uint32_t present[128];
  __shared__ uint32_t small[3][8 * 128];   // short vanishing polynomial, its DFT on <nu>, its DFT on 7^64 <nu>
  const int blob = blockIdx.x, tid = threadIdx.x;
  const int fail = mode == 0 ? 2 : 1;
  coef_out += (size_t)blob * 4096;
  ws += (size_t)blob * 3 * 8192;
  evals += (size_t)blob * n_cells * CELL_ELEMS * 8;
  cell_status += (size_t)blob * n_cells;
  cell_indices += (size_t)blob * n_cells;
  Fr* ext = ws;              // E in natural order, later E * Z, later the quotient
  Fr* tmp = ws + 8192;
  Fr* tmp2 = ws + 16384;
  if (tid < 128) present[tid] = 0;
  bool malformed = false;
  if (tid < n_cells) {
    const uint64_t ix = cell_indices[tid];
    malformed = ix >= N_CELLS || (tid > 0 && ix <= cell_indices[tid - 1]) || cell_status[tid] != 0;
  }
  if (__syncthreads_or(malformed)) {
    for (int i = tid; i < 4096; i += blockDim.x) coef_out[i] = fr_zero();
    if (tid == 0) status[blob] = fail;
    return;
  }
  if (tid < n_cells) present[cell_indices[tid] & 127u] = 1;
  __syncthreads();
  // ---- short vanishing polynomial prod (X - nu^brp7(i)) over the missing cells i (degree <= 64), by one thread
  if (tid == 0) {
    for (int d = 0; d < 128; d++) sm_store<128>(small[0], d, d == 0 ? fr_one() : fr_zero());
    int deg = 0;
    for (int i = 0; i < 128; i++) {
      if (present[i]) continue;
      const Fr root = tw[64u * brp7(i)];
      // multiply by (X - root): new[d] = old[d-1] - root * old[d]
      Fr prev = fr_zero();
      for (int d = 0; d <= deg + 1; d++) {
        const Fr cur = sm_load<128>(small[0], d);
        sm_store<128>(small[0], d, fr_sub(prev, fr_mul(root, cur)));
        prev = cur;
      }
      deg++;
    }
  }
  // ---- E in natural order: ext[brp13(64 ci + j)] = cell value j of cell ci; zero where missing
  for (int i = tid; i < 8192; i += blockDim.x) ext[i] = fr_zero();
  __syncthreads();
  for (int t = tid; t < n_cells * 64; t += blockDim.x) {
    const int kq = t / 64, j = t % 64;
    const uint32_t pos = (uint32_t)(cell_indices[kq] & 127u) * 64u + j;
    Fr v;
    for (int l = 0; l < 8; l++) v.l[l] = evals[(size_t)t * 8 + l];
    ext[__brev(pos) >> 19] = fr_to_mont(v);
  }
  // ---- Z on the domain and on the coset: Z(X) = short(X^64), so Z(w8192^k) = short(nu^k) has period 128, and
  // Z(7 w8192^k) = short(7^64 nu^k): two 128-point DFTs of short_d and short_d 7^(64 d)
  __syncthreads();
  {
    Fr seven = fr_zero();
    seven.l[0] = 7;
    const Fr s64 = fr_pow_small(fr_to_mont(seven), 64);
    for (int d = tid; d < 128; d += blockDim.x) {
      const Fr v = sm_load<128>(small[0], d);
      sm_store<128>(small[1], d, v);
      sm_store<128>(small[2], d, fr_mul(v, fr_pow_small(s64, (uint32_t)d)));
    }
  }
  __syncthreads();
  sm_dif<128>(small[1], tw, false);   // position p holds short(nu^brp7(p))
  sm_dif<128>(small[2], tw, false);
  // ---- (E Z) on the domain -> coefficients
  for (int i = tid; i < 8192; i += blockDim.x) ext[i] = fr_mul(ext[i], sm_load<128>(small[1], brp7(i & 127)));
  __syncthreads();
  fft8192(tmp, ext, sm, tw, true);    // unscaled inverse: 8192 * (E Z) coefficients
  // ---- to the coset: multiply coefficient n by 7^n (and by 1/8192), forward transform, divide by Z on the coset
  {
    Fr seven = fr_zero();
    seven.l[0] = 7;
    const Fr s = fr_to_mont(seven);
    Fr n_inv = fr_const(k::FR_N_INV);   // 1/4096
    Fr two = fr_add(fr_one(), fr_one());
    n_inv = fr_mul(n_inv, fr_inv(two));  // 1/8192
    // each thread walks a contiguous run of 16 exponents
    const int base = tid * 16;
    Fr p = fr_mul(fr_pow_small(s, (uint32_t)base), n_inv);
    for (int u = 0; u < 16; u++) {
      tmp[base + u] = fr_mul(tmp[base + u], p);
      p = fr_mul(p, s);
    }
  }
  __syncthreads();
  fft8192(tmp2, tmp, sm, tw, false);
  // 128 distinct denominators: invert each (Fermat; 128 threads)
  if (tid < 128) sm_store<128>(small[0], tid, fr_inv(sm_load<128>(small[2], tid)));
  __syncthreads();
  for (int i = tid; i < 8192; i += blockDim.x) tmp2[i] = fr_mul(tmp2[i], sm_load<128>(small[0], brp7(i & 127)));
  __syncthreads();
  fft8192(tmp, tmp2, sm, tw, true);
  // ---- back from the coset: coefficient n times 7^-n / 8192; the upper half must vanish
  {
    Fr seven = fr_zero();
    seven.l[0] = 7;
    const Fr sinv = fr_inv(fr_to_mont(seven));
    Fr n_inv = fr_const(k::FR_N_INV);
    Fr two = fr_add(fr_one(), fr_one());
    n_inv = fr_mul(n_inv, fr_inv(two));
    const int base = tid * 16;
    Fr p = fr_mul(fr_pow_small(sinv, (uint32_t)base), n_inv);
    bool bad = false;
    for (int u = 0; u < 16; u++) {
      const Fr v = fr_mul(tmp[base + u], p);
      if (base + u < 4096) coef_out[base + u] = v;
      else if (!fr_is_zero(v)) bad = true;
      p = fr_mul(p, sinv);
    }
    // inconsistent cells: no polynomial of degree < 4096 matches them
    bad = __syncthreads_or(bad);
    if (tid == 0) status[blob] = bad ? fail : 0;
  }
}

}  // namespace

void launch_cell_parse(void* d_evals, int* d_status, const void* d_cells, int n_cells, int mode, cudaStream_t st) {
  if (n_cells <= 0) return;
  const long total = (long)n_cells * CELL_ELEMS;
  LW_SAME_CARVEOUT(cell_parse_kernel);
  cell_parse_kernel<<<(unsigned)((total + 127) / 128), 128, 0, st>>>((uint32_t*)d_evals, d_status, (const uint8_t*)d_cells, n_cells, mode);
  count_launch();
}

void launch_cell_batch_challenge(void* d_r, const void* d_commitments48, int n_commitments, const uint32_t* d_commitment_indices, const uint64_t* d_cell_indices,
                                 const void* d_cells, const void* d_proofs48, int n_cells, int mode, cudaStream_t st) {
  CellMsg m;
  m.commitments = (const uint32_t*)d_commitments48;
  m.commitment_indices = d_commitment_indices;
  m.cell_indices = d_cell_indices;
  m.cells = (const uint32_t*)d_cells;
  m.proofs = (const uint32_t*)d_proofs48;
  m.n_commitments = (unsigned long long)n_commitments;
  m.n_cells = (unsigned long long)n_cells;
  m.le = mode == 1 ? 1 : 0;
  m.uniq = nullptr;
  m.set_head();
  LW_SAME_CARVEOUT(cell_batch_challenge_kernel);
  cell_batch_challenge_kernel<<<1, 32, 0, st>>>((uint32_t*)d_r, m);
  count_launch();
}

void launch_cell_verify_scalars(void* d_wcoef, void* d_rpow, void* d_scalars_b, const void* d_evals, const uint64_t* d_cell_indices,
                                const uint32_t* d_commitment_indices, int n_cells, int n_commitments, const void* d_r, const void* d_tw8192, cudaStream_t st) {
  if (n_cells <= 0) return;
  LW_SAME_CARVEOUT(cell_interp_kernel<false>);
  LW_SAME_CARVEOUT(cell_verify_finish_kernel);
  cell_interp_kernel<false><<<n_cells, 32, 0, st>>>((Fr*)d_wcoef, (uint32_t*)d_rpow, (uint32_t*)d_scalars_b, (const uint32_t*)d_evals, d_cell_indices,
                                                   (const uint32_t*)d_r, (const Fr*)d_tw8192, nullptr, nullptr);
  cell_verify_finish_kernel<<<1, 128, 0, st>>>((uint32_t*)d_scalars_b, (const Fr*)d_wcoef, (const uint32_t*)d_rpow, d_commitment_indices, n_cells, n_commitments);
  count_launch(2);
}

void launch_cell_recover(void* d_coef, int* d_status, void* d_ws, const void* d_evals, const int* d_cell_status, const uint64_t* d_cell_indices,
                         int n_blobs, int n_cells, int mode, const void* d_tw8192, cudaStream_t st) {
  if (n_blobs <= 0) return;
  static bool attr_set[64] = {};   // function attributes are per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 64 && !attr_set[dev]) {
    cudaFuncSetAttribute(cell_recover_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, REC_SMEM);
    attr_set[dev] = true;
  }
  cell_recover_kernel<<<n_blobs, REC_THREADS, REC_SMEM, st>>>((Fr*)d_coef, d_status, (Fr*)d_ws, (const uint32_t*)d_evals, d_cell_status, d_cell_indices,
                                                             n_cells, mode, (const Fr*)d_tw8192);
  count_launch();
}

void launch_cell_batches_prepare(int* d_bstatus, int* d_nc, uint32_t* d_cidx, uint32_t* d_uniq, int* d_first, int* d_cell_batch, const void* d_commit48,
                                 const uint64_t* d_cell_indices, const int* d_cell_status, int n_cells, const int* d_boff, int nb, int mode, cudaStream_t st) {
  if (nb <= 0) return;
  cell_batches_prepare_kernel<<<nb, 256, 0, st>>>(d_bstatus, d_nc, d_cidx, d_uniq, d_first, d_cell_batch, (const uint8_t*)d_commit48, d_cell_indices, d_cell_status,
                                                  n_cells, d_boff, mode);
  count_launch();
}

void launch_cell_batches_challenge(void* d_rs, const void* d_commit48, const uint32_t* d_uniq, const uint32_t* d_cidx, const uint64_t* d_cell_indices,
                                   const void* d_cells, const void* d_proofs48, const int* d_nc, const int* d_boff, int nb, int mode, cudaStream_t st) {
  if (nb <= 0) return;
  LW_SAME_CARVEOUT(cell_batches_challenge_kernel);
  cell_batches_challenge_kernel<<<nb, 32, 0, st>>>((uint32_t*)d_rs, (const uint32_t*)d_commit48, d_uniq, d_cidx, d_cell_indices, (const uint32_t*)d_cells,
                                                   (const uint32_t*)d_proofs48, d_nc, d_boff, mode == 1 ? 1 : 0);
  count_launch();
}

void launch_cell_batches_scalars(void* d_wcoef, void* d_scal, const void* d_evals, const uint64_t* d_cell_indices, const uint32_t* d_cidx, const int* d_nc,
                                 const int* d_cell_batch, const int* d_boff, int n_cells, int nb, const void* d_rs, const void* d_tw8192, cudaStream_t st) {
  if (nb <= 0) return;
  if (n_cells > 0) {
    LW_SAME_CARVEOUT(cell_interp_kernel<true>);
    cell_interp_kernel<true><<<n_cells, 32, 0, st>>>((Fr*)d_wcoef, (uint32_t*)d_scal, (uint32_t*)d_scal, (const uint32_t*)d_evals, d_cell_indices,
                                                    (const uint32_t*)d_rs, (const Fr*)d_tw8192, d_cell_batch, d_boff);
    count_launch();
  }
  cell_batches_finish_kernel<<<nb, 128, 0, st>>>((uint32_t*)d_scal, (const Fr*)d_wcoef, d_cidx, d_nc, d_boff);
  count_launch();
}

size_t cell_segmsm_terms(int n_cells, int nb) { return cell_batch_term_base(n_cells, nb); }

void launch_cell_segmsm(void* d_out288, void* d_terms, const void* d_scal, const void* d_proof_aff, const void* d_commit_aff, const void* d_mono_aff,
                        const uint32_t* d_uniq, const int* d_nc, const int* d_boff, int n_cells, int nb, cudaStream_t st) {
  if (nb <= 0) return;
  const long n_terms = (long)cell_segmsm_terms(n_cells, nb);
  cell_segmsm_terms_kernel<<<(unsigned)((n_terms + 127) / 128), 128, 0, st>>>((G1Xyzz*)d_terms, (const uint32_t*)d_scal, (const G1Affine*)d_proof_aff,
                                                                             (const G1Affine*)d_commit_aff, (const G1Affine*)d_mono_aff, d_uniq, d_nc, d_boff,
                                                                             nb, n_terms);
  cell_segmsm_reduce_kernel<<<2 * nb, 128, 0, st>>>((uint8_t*)d_out288, (const G1Xyzz*)d_terms, d_boff);
  count_launch(2);
}

void launch_cell_blob_broadcast(void* d_commit48, void* d_commit_aff, int* d_commit_status, uint64_t* d_cell_indices, const void* d_blob_commit48,
                                const void* d_blob_aff, const int* d_blob_status, int n_blobs, cudaStream_t st) {
  if (n_blobs <= 0) return;
  cell_blob_broadcast_kernel<<<n_blobs, N_CELLS, 0, st>>>((uint8_t*)d_commit48, (G1Affine*)d_commit_aff, d_commit_status, d_cell_indices,
                                                          (const uint8_t*)d_blob_commit48, (const G1Affine*)d_blob_aff, d_blob_status, n_blobs);
  count_launch();
}

void launch_fill_int(int* d_out, int value, int n, cudaStream_t st) {
  if (n <= 0) return;
  fill_int_kernel<<<(n + 127) / 128, 128, 0, st>>>(d_out, value, n);
  count_launch();
}

void launch_cell_batches_fold(int* d_ok, int* d_status, const int* d_pair_ok, const int* d_bstatus, const int* d_boff, int nb, cudaStream_t st) {
  if (nb <= 0) return;
  cell_batches_fold_kernel<<<(nb + 127) / 128, 128, 0, st>>>(d_ok, d_status, d_pair_ok, d_bstatus, d_boff, nb);
  count_launch();
}

}  // namespace lw
