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
  const uint32_t* commitment_indices;
  const uint64_t* cell_indices;
  const uint32_t* cells;         // 512 words each
  const uint32_t* proofs;        // 12 words each
  uint32_t head[12];
  unsigned long long n_commitments, n_cells;
  int le;                        // little-endian integers (MODE_CKZG_LE)
  __device__ __forceinline__ void u64_words(uint32_t* out2, unsigned long long v) const {
    if (le) { out2[0] = bswap32((uint32_t)v); out2[1] = bswap32((uint32_t)(v >> 32)); }
    else { out2[0] = (uint32_t)(v >> 32); out2[1] = (uint32_t)v; }
  }
  __device__ __forceinline__ unsigned long long total_words() const { return 12ull + 12ull * n_commitments + 528ull * n_cells; }
  __device__ __forceinline__ uint32_t word(unsigned long long wi) const {
    if (wi < 12) return head[wi];
    wi -= 12;
    if (wi < 12ull * n_commitments) return bswap32(__ldg(commitments + wi));
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

__global__ void __launch_bounds__(32) cell_batch_challenge_kernel(uint32_t* __restrict__ r_out, CellMsg msg) {
  __shared__ uint32_t wk[64 * 32];
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

// ------------------------------------------------------------------ scalars of the two MSMs
// One warp per cell: a = IDFT_64 of the cell's evaluations (given in bit-reversed order), coefficient m of the
// interpolation polynomial = a_m h^-m / 64; weighted by r^k and written to wcoef[k][m] (Montgomery).
// Lane 0 also writes r^k (rpow, canonical) and r^k h^64 (scalars_b[k], canonical).
__global__ void __launch_bounds__(32) cell_interp_kernel(Fr* __restrict__ wcoef, uint32_t* __restrict__ rpow, uint32_t* __restrict__ scalars_b,
                                                        const uint32_t* __restrict__ evals, const uint64_t* __restrict__ cell_indices,
                                                        const uint32_t* __restrict__ r_canon, const Fr* __restrict__ tw) {
  __shared__ uint32_t sm[8 * 64];
  const int kq = blockIdx.x, lane = threadIdx.x;
  const uint32_t hexp = brp7((uint32_t)cell_indices[kq] & 127u);   // h_k = w8192^brp7(cell index)
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = r_canon[i];
  const Fr rk = fr_pow_small(fr_to_mont(r), (uint32_t)kq);
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
    for (int l = 0; l < 8; l++) { rpow[(size_t)kq * 8 + l] = a.l[l]; scalars_b[(size_t)kq * 8 + l] = b.l[l]; }
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
  const char dom[17] = "RCKZGCBATCH__V1_";
  for (int i = 0; i < 4; i++)
    m.head[i] = ((uint32_t)(uint8_t)dom[4 * i] << 24) | ((uint32_t)(uint8_t)dom[4 * i + 1] << 16) | ((uint32_t)(uint8_t)dom[4 * i + 2] << 8) | (uint32_t)(uint8_t)dom[4 * i + 3];
  auto put = [&](int at, unsigned long long v) {
    if (m.le) { m.head[at] = __builtin_bswap32((uint32_t)v); m.head[at + 1] = __builtin_bswap32((uint32_t)(v >> 32)); }
    else { m.head[at] = (uint32_t)(v >> 32); m.head[at + 1] = (uint32_t)v; }
  };
  put(4, 4096);
  put(6, CELL_ELEMS);
  put(8, m.n_commitments);
  put(10, m.n_cells);
  LW_SAME_CARVEOUT(cell_batch_challenge_kernel);
  cell_batch_challenge_kernel<<<1, 32, 0, st>>>((uint32_t*)d_r, m);
  count_launch();
}

void launch_cell_verify_scalars(void* d_wcoef, void* d_rpow, void* d_scalars_b, const void* d_evals, const uint64_t* d_cell_indices,
                                const uint32_t* d_commitment_indices, int n_cells, int n_commitments, const void* d_r, const void* d_tw8192, cudaStream_t st) {
  if (n_cells <= 0) return;
  LW_SAME_CARVEOUT(cell_interp_kernel);
  LW_SAME_CARVEOUT(cell_verify_finish_kernel);
  cell_interp_kernel<<<n_cells, 32, 0, st>>>((Fr*)d_wcoef, (uint32_t*)d_rpow, (uint32_t*)d_scalars_b, (const uint32_t*)d_evals, d_cell_indices,
                                            (const uint32_t*)d_r, (const Fr*)d_tw8192);
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

}  // namespace lw
