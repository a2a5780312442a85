// Verification kernels: single-proof check, random-linear-combination batch
// check and the generic G1 linear combination.
//   verify_kzg_proof / verify_blob_kzg_proof     /root/reference/src/lib.rs:407-505
//   verify_blob_kzg_proof_batch / verify_kzg_proof_batch          src/lib.rs:525-692
//   compute_r_powers                                              src/utils.rs:156-206
//   g1_lincomb                                                    src/lib.rs:241-243
// The pairing equation e(C - y g1[0], g2[0]) e(-pi, g2[1] - z g2[0]) == 1 is
// evaluated in the bilinearly equivalent form
//        e(C - y g1[0] + z pi, g2[0]) * e(-pi, g2[1]) == 1
// so that both G2 arguments are the FIXED setup points whose Miller-loop lines
// were precomputed at load time (pairing.cuh): no G2 arithmetic at verify time.
#include <algorithm>

#include "kernels.h"
#include "batch_challenge.cuh"
#include "pairing_warp.cuh"
#include "sha256.cuh"

namespace lw {

struct G2PreparedDev {
  G2Prepared p;
};
size_t g2_prepared_bytes() { return sizeof(G2Prepared); }

// canonical x.c0,x.c1,y.c0,y.c1 -> prepared lines.  bad = 1 if the point is not
// on the twist (blst_p2_to_g2_point's from_affine, src/srs.rs:215-247; the
// all-zero encoding of infinity fails that check too).  One point per block.
__global__ void g2_prepare_kernel(G2Prepared* __restrict__ out, int* __restrict__ bad, const uint32_t* __restrict__ canon48) {
  if (threadIdx.x != 0) return;
  out += blockIdx.x;
  bad += blockIdx.x;
  canon48 += (size_t)blockIdx.x * 48;
  Fp c[4];
  for (int j = 0; j < 4; j++) {
    for (int k = 0; k < 12; k++) c[j].l[k] = canon48[j * 12 + k];
    mod_reduce_small<FpCfg, 9>(c[j].l);
    c[j] = fp_to_mont(c[j]);
  }
  G2Affine q;
  q.x.c0 = c[0]; q.x.c1 = c[1]; q.y.c0 = c[2]; q.y.c1 = c[3];
  if (!g2a_on_curve(q)) { *bad = 1; out->infinity = 1; return; }
  *bad = 0;
  g2_prepare(*out, q);
}

// on-curve check of all 65 g2 values (the reference re-hydrates -- and so
// validates -- every one of them on every call: src/srs.rs:258-280)
__global__ void g2_check_kernel(int* __restrict__ bad, const uint32_t* __restrict__ canon48, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp c[4];
  for (int j = 0; j < 4; j++) {
    for (int k = 0; k < 12; k++) c[j].l[k] = canon48[i * 48 + j * 12 + k];
    mod_reduce_small<FpCfg, 9>(c[j].l);
    c[j] = fp_to_mont(c[j]);
  }
  G2Affine q;
  q.x.c0 = c[0]; q.x.c1 = c[1]; q.y.c0 = c[2]; q.y.c1 = c[3];
  bad[i] = g2a_on_curve(q) ? 0 : 1;
}

// ---- two-pairing check, block-cooperative (pairing_warp.cuh): every Fp12 product is
// spread over the lanes.  `pts` (2 points) and `m` live in shared memory; all
// LW_PAIR_LANES threads of the block must call this.
__device__ __forceinline__ bool two_pairing_check(const G1Affine* pts, const G2Prepared* prep0, const G2Prepared* prep1, WarpPairingMem& m) {
  const G2Prepared* qs[2] = {prep0, prep1};
  warp_pairing_product(m, pts, qs, 2);
  bool ok = false;
  if (threadIdx.x == 0) ok = warp_fp12_is_one(m.f);
  return ok;
}

// ok = [ e(C - y g1_0 + z pi, g2_0) * e(-pi, g2_1) == 1 ]
// Block of VS_THREADS = 160: warps 0-1 are the pairing group (LW_PAIR_LANES); before that, lane 0 of each of the
// warps 0..3 runs one of the four GLV half-ladders and lanes 0-1 of warp 4 the two r-torsion tests.  One ladder per
// WARP, not four in one warp: the lanes of a warp execute every conditional addition any of them needs (94 % of the
// bits for four random scalars instead of 50 %), so sharing a warp made each ladder cost 128 doublings + 120 additions.
constexpr int VS_THREADS = 160;
__global__ void __launch_bounds__(VS_THREADS) verify_single_kernel(int* __restrict__ ok_out, const G1Affine* __restrict__ c_aff, const G1Affine* __restrict__ pi_aff,
                                                            const uint32_t* __restrict__ z, const uint32_t* __restrict__ y,
                                                            const G1Affine* __restrict__ g1_0, const G2Prepared* __restrict__ prep0,
                                                            const G2Prepared* __restrict__ prep1, int g1_0_in_subgroup, int* __restrict__ status,
                                                            int sub_code) {
  __shared__ G1Xyzz sh_pt[4];
  __shared__ WarpPairingMem sh_m;
  __shared__ G1Affine sh_pair[2];
  const int lane = threadIdx.x;
  G1Affine C = *c_aff, PI = *pi_aff;
  if (lane < 128 && (lane & 31) == 0) {
    // four warps share the two scalar multiplications: GLV halves k = q x^2 + m, [k]P = [m]P + [q](beta x, -y)
    // (z and y are canonical, < r), 128 doublings each instead of 255
    const int job = lane >> 5;
    const int which = job >> 1, half = job & 1;
    uint32_t k[8], q[4], m[4];
    for (int i = 0; i < 8; i++) k[i] = which == 0 ? y[i] : z[i];
    glv_split(q, m, k);
    G1Affine base = which == 0 ? *g1_0 : PI;
    // phi(P) = [-x^2]P holds on the r-torsion only: pi is subgroup-checked (when decoded, or beside this ladder), a
    // hand-built setup's g1[0] need not be (srs.rs:155-172 checks the curve equation only) -> plain 255-bit ladder
    const bool glv = which == 1 || g1_0_in_subgroup != 0;
    if (!glv) {
      sh_pt[job] = half == 0 ? g1_mul_scalar(base, k, 8) : xyzz_inf();
    } else {
      if (half == 1 && !g1a_is_inf(base)) {
        Fp beta;
        for (int i = 0; i < 12; i++) beta.l[i] = k::FP_BETA[i];
        base.x = fp_mul(base.x, beta);
        base.y = fp_neg(base.y);
      }
      sh_pt[job] = g1_mul_scalar(base, half == 0 ? m : q, 4);
    }
  }
  // sub_code != 0: C and pi were decoded WITHOUT the r-torsion test (the larger part of a decompression); two lanes
  // of the fifth warp run it here, beside the scalar multiplications instead of in front of them.
  // A failure is reported through status[0] and overrides whatever the pairing says.
  if (sub_code != 0 && (lane == 128 || lane == 129)) {
    if (!g1_in_subgroup(lane == 128 ? C : PI)) atomicCAS(status, 0, sub_code);
  }
  __syncthreads();
  if (lane == 0) {
    G1Xyzz acc = xyzz_from_affine(C);
    G1Xyzz yg = sh_pt[0];
    xyzz_add_ni(yg, sh_pt[1]);
    xyzz_add_ni(acc, xyzz_neg(yg));
    xyzz_add_ni(acc, sh_pt[2]);
    xyzz_add_ni(acc, sh_pt[3]);
    sh_pair[0] = xyzz_to_affine(acc);
    sh_pair[1] = g1a_neg(PI);
  }
  __syncthreads();
  bool ok = two_pairing_check(sh_pair, prep0, prep1, sh_m);
  if (lane == 0) *ok_out = ok ? 1 : 0;
}

// tuple_i = compress(C_i) || be32(z_i) || be32(y_i) || compress(pi_i)  (utils.rs:183-201)
__global__ void make_tuples_kernel(uint8_t* __restrict__ tuples, const uint8_t* __restrict__ c48, const uint32_t* __restrict__ z,
                                   const uint32_t* __restrict__ y, const uint8_t* __restrict__ pi48, int n, int le) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t* t = tuples + (size_t)i * 160;
  for (int k = 0; k < 48; k++) t[k] = c48[(size_t)i * 48 + k];
  Fr zz, yy;
  for (int k = 0; k < 8; k++) { zz.l[k] = z[i * 8 + k]; yy.l[k] = y[i * 8 + k]; }
  if (le) {  // MODE_CKZG_LE: field elements are hashed little-endian
    for (int k = 0; k < 8; k++)
      for (int b = 0; b < 4; b++) { t[48 + 4 * k + b] = (uint8_t)(zz.l[k] >> (8 * b)); t[80 + 4 * k + b] = (uint8_t)(yy.l[k] >> (8 * b)); }
  } else {
    fr_canon_to_be32(t + 48, zz);
    fr_canon_to_be32(t + 80, yy);
  }
  for (int k = 0; k < 48; k++) t[112 + k] = pi48[(size_t)i * 48 + k];
}

// The batch challenge over one batch (batch_challenge.cuh).  Its input becomes available chunk by chunk while a batch
// is being prepared (tuple i exists as soon as blob i has been copied, hashed and evaluated), so the kernel works on a
// block range of the message: [blk0, blk1) 64-byte blocks, state carried in `state` between launches.  One launch with
// BCH_INIT | BCH_FINAL and blk0 = blk1 = 0 is the monolithic hash.
__global__ void __launch_bounds__(32) batch_challenge_kernel(uint32_t* __restrict__ r_out, Sha256State* __restrict__ state, const uint8_t* __restrict__ tuples,
                                                              unsigned long long n_total, int blk0, int blk1, int flags) {
  __shared__ uint32_t wk[64 * 32];
  __shared__ uint8_t head[32];
  batch_challenge_warp(r_out, state, tuples, n_total, blk0, blk1, flags, wk, head);
}

// XYZZ block reduction helpers (same SoA shared-memory layout as msm.cu)
__device__ __forceinline__ void xyzz_to_smem(uint32_t* smem, int stride, int t, const G1Xyzz& p) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&p);
#pragma unroll
  for (int i = 0; i < 48; i++) smem[i * stride + t] = w[i];
}
__device__ __forceinline__ G1Xyzz xyzz_from_smem(const uint32_t* smem, int stride, int t) {
  G1Xyzz p;
  uint32_t* w = reinterpret_cast<uint32_t*>(&p);
#pragma unroll
  for (int i = 0; i < 48; i++) w[i] = smem[i * stride + t];
  return p;
}
template <int THREADS>
__device__ __forceinline__ void block_reduce_xyzz(G1Xyzz& acc, uint32_t* red) {
  const int tid = threadIdx.x;
  for (int s = THREADS / 2; s > 0; s >>= 1) {
    if (tid >= s && tid < 2 * s) xyzz_to_smem(red, THREADS / 2, tid - s, acc);
    __syncthreads();
    if (tid < s) {
      G1Xyzz o = xyzz_from_smem(red, THREADS / 2, tid);
      xyzz_add_ni(acc, o);
    }
    __syncthreads();
  }
}

// ---- the random linear combination of a batched verification (verify_kzg_proof_batch, lib.rs:639-692) as two
// bucket MSMs over the batch -- the reference computes it with three `msm` calls (lib.rs:679-685):
//   proof_lincomb                        = sum r^i pi_i                                   (n points)
//   proof_z_lincomb + c_minus_y_lincomb  = sum (r^i z_i) pi_i + sum r^i C_i - (sum r^i y_i) G   (2n + 1 points)
// (the pairing check only ever uses the SUM of the last two).  This kernel derives the scalars and lays the
// points of the second MSM out contiguously: [C_0 .. C_{n-1} | pi_0 .. pi_{n-1} | G].
constexpr int RLC_THREADS = 128;
__global__ void __launch_bounds__(RLC_THREADS) rlc_scalars_kernel(uint32_t* __restrict__ sc_a, uint32_t* __restrict__ sc_b, G1Affine* __restrict__ pts_b,
                                                                   uint32_t* __restrict__ ypart, uint32_t* __restrict__ ticket,
                                                                   const uint32_t* __restrict__ r_in, const G1Affine* __restrict__ c_aff,
                                                                   const G1Affine* __restrict__ pi_aff, const uint32_t* __restrict__ z,
                                                                   const uint32_t* __restrict__ y, unsigned long long first, int n) {
  __shared__ uint32_t ysum[RLC_THREADS][8];
  __shared__ bool is_last;
  const int i = blockIdx.x * RLC_THREADS + threadIdx.x;
  Fr ys = fr_zero();   // canonical r^(first + i) y_i
  if (i < n) {
    Fr rc;
    for (int k = 0; k < 8; k++) rc.l[k] = r_in[k];
    const Fr rm = fr_to_mont(rc);
    const unsigned long long e = first + (unsigned long long)i;
    Fr pw = fr_one();   // r^e, Montgomery
    bool started = false;
    for (int bit = 63; bit >= 0; bit--) {
      if (started) pw = fr_sqr(pw);
      if ((e >> bit) & 1ull) { pw = fr_mul(pw, rm); started = true; }
    }
    Fr zc, yc;
    for (int k = 0; k < 8; k++) { zc.l[k] = z[i * 8 + k]; yc.l[k] = y[i * 8 + k]; }
    const Fr p1 = fr_from_mont(pw);
    const Fr pz = fr_mul(pw, zc);   // mont(r^e) * canonical z = canonical r^e z
    ys = fr_mul(pw, yc);
    for (int k = 0; k < 8; k++) {
      sc_a[(size_t)i * 8 + k] = p1.l[k];
      sc_b[(size_t)i * 8 + k] = p1.l[k];
      sc_b[((size_t)n + i) * 8 + k] = pz.l[k];
    }
    pts_b[i] = c_aff[i];
    pts_b[(size_t)n + i] = pi_aff[i];
  }
  for (int k = 0; k < 8; k++) ysum[threadIdx.x][k] = ys.l[k];
  __syncthreads();
  for (int s = RLC_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      Fr a, b;
      for (int k = 0; k < 8; k++) { a.l[k] = ysum[threadIdx.x][k]; b.l[k] = ysum[threadIdx.x + s][k]; }
      a = fr_add(a, b);
      for (int k = 0; k < 8; k++) ysum[threadIdx.x][k] = a.l[k];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    for (int k = 0; k < 8; k++) ypart[(size_t)blockIdx.x * 8 + k] = ysum[0][k];
    __threadfence();
    is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last || threadIdx.x != 0) return;
  // last block: - (sum r^i y_i) times the generator G (lib.rs:661-668 uses the curve generator)
  __threadfence();
  Fr tot = fr_zero();
  for (unsigned b = 0; b < gridDim.x; b++) {
    Fr v;
    for (int k = 0; k < 8; k++) v.l[k] = __ldcg(ypart + (size_t)b * 8 + k);
    tot = fr_add(tot, v);
  }
  tot = fr_neg(tot);
  for (int k = 0; k < 8; k++) sc_b[(size_t)2 * n * 8 + k] = tot.l[k];
  pts_b[(size_t)2 * n] = g1a_generator();
  *ticket = 0;
}

__device__ __forceinline__ G1Affine affine_from_be96(const uint8_t* b) {
  bool z = true;
  for (int k = 0; k < 96; k++) z = z && (b[k] == 0);
  if (z) return g1a_inf();
  G1Affine p;
  p.x = fp_from_be48(b);
  p.y = fp_from_be48(b + 48);
  return p;
}

// partials: n_ranks x (proof_lincomb, proof_z_lincomb, c_minus_y_lincomb), canonical BE affine.
// ok = [ e(c_minus_y + proof_z, g2_0) == e(proof_lincomb, g2_1) ]   (lib.rs:679-691)
// Block b checks the partials at b * n_ranks * 288 against prep0 + b * prep_stride, prep1 + b * prep_stride.
__global__ void __launch_bounds__(LW_PAIR_LANES) batch_final_kernel(int* __restrict__ ok_out, const uint8_t* __restrict__ partials, int n_ranks,
                                                          const G2Prepared* __restrict__ prep0, const G2Prepared* __restrict__ prep1, int prep_stride) {
  __shared__ WarpPairingMem sh_m;
  __shared__ G1Affine sh_pts[2];
  const int lane = threadIdx.x;
  partials += (size_t)blockIdx.x * n_ranks * 288;   // one check per block (launch_batch_final_each)
  ok_out += blockIdx.x;
  prep0 += (size_t)blockIdx.x * prep_stride;
  prep1 += (size_t)blockIdx.x * prep_stride;
  if (lane < 2) {
    G1Xyzz acc = xyzz_inf();
    for (int r = 0; r < n_ranks; r++) {
      const uint8_t* base = partials + (size_t)r * 288;
      if (lane == 0) {
        xyzz_madd_ni(acc, affine_from_be96(base + 96));   // proof_z_lincomb
        xyzz_madd_ni(acc, affine_from_be96(base + 192));  // c_minus_y_lincomb
      } else {
        xyzz_madd_ni(acc, affine_from_be96(base));        // proof_lincomb
      }
    }
    G1Affine a = xyzz_to_affine(acc);
    sh_pts[lane] = lane == 0 ? a : g1a_neg(a);
  }
  __syncthreads();
  bool ok = two_pairing_check(sh_pts, prep0, prep1, sh_m);
  if (lane == 0) *ok_out = ok ? 1 : 0;
}

// ------------------------------------------------------------------ launchers
void launch_g2_prepare(void* d_prepared, int* d_bad, const void* d_canon_in, cudaStream_t st, int n) {
  if (n <= 0) return;
  g2_prepare_kernel<<<n, 32, 0, st>>>((G2Prepared*)d_prepared, d_bad, (const uint32_t*)d_canon_in);
  count_launch();
}
void launch_g2_check(int* d_bad, const void* d_canon_in, int n, cudaStream_t st) {
  g2_check_kernel<<<(n + 31) / 32, 32, 0, st>>>(d_bad, (const uint32_t*)d_canon_in, n);
  count_launch();
}
void launch_verify_single(int* d_ok, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y, const void* d_g1_0_aff,
                          const void* d_prep0, const void* d_prep1, bool g1_0_in_subgroup, cudaStream_t st, int* d_status, int sub_code) {
  verify_single_kernel<<<1, VS_THREADS, 0, st>>>(d_ok, (const G1Affine*)d_c_aff, (const G1Affine*)d_pi_aff, (const uint32_t*)d_z, (const uint32_t*)d_y,
                                         (const G1Affine*)d_g1_0_aff, (const G2Prepared*)d_prep0, (const G2Prepared*)d_prep1, g1_0_in_subgroup ? 1 : 0,
                                         d_status, d_status ? sub_code : 0);
  count_launch();
}
void launch_make_tuples(void* d_tuples160, const void* d_c48, const void* d_z, const void* d_y, const void* d_pi48, int n, cudaStream_t st, bool le) {
  if (n <= 0) return;
  LW_SAME_CARVEOUT(make_tuples_kernel);
  make_tuples_kernel<<<(n + 63) / 64, 64, 0, st>>>((uint8_t*)d_tuples160, (const uint8_t*)d_c48, (const uint32_t*)d_z, (const uint32_t*)d_y, (const uint8_t*)d_pi48, n,
                                                  le ? 1 : 0);
  count_launch();
}
// (measured and not kept: giving this one-warp kernel an SM of its own by asking for all of the SM's shared memory --
// no change; what slowed the device-resident batch was eight chunk streams at once, see "verify_streams")
void launch_batch_challenge(void* d_r, const void* d_tuples160, size_t n_total, cudaStream_t st, int wire) {
  LW_SAME_CARVEOUT(batch_challenge_kernel);
  batch_challenge_kernel<<<1, 32, 0, st>>>((uint32_t*)d_r, nullptr, (const uint8_t*)d_tuples160, (unsigned long long)n_total, 0, 0,
                                                              BCH_INIT | BCH_FINAL | bch_wire_flags(wire));
  count_launch();
}
size_t batch_challenge_state_bytes() { return sizeof(Sha256State); }
int batch_challenge_blocks_ready(size_t tuples_ready) { return (int)((32 + 160 * tuples_ready) / 64); }
void launch_batch_challenge_part(void* d_r, void* d_state, const void* d_tuples160, size_t n_total, int blk0, int blk1, bool first, bool last,
                                 cudaStream_t st, int wire) {
  if (!last && blk1 <= blk0 && !first) return;
  LW_SAME_CARVEOUT(batch_challenge_kernel);
  batch_challenge_kernel<<<1, 32, 0, st>>>((uint32_t*)d_r, (Sha256State*)d_state, (const uint8_t*)d_tuples160, (unsigned long long)n_total,
                                                              blk0, blk1, (first ? BCH_INIT : 0) | (last ? BCH_FINAL : 0) | bch_wire_flags(wire));
  count_launch();
}
struct RlcLayout { size_t sc_a, sc_b, pts_b, ypart, ticket, msm_a, msm_b, total; };
static RlcLayout rlc_layout(size_t n) {
  RlcLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
  const size_t blocks = (n + RLC_THREADS - 1) / RLC_THREADS + 1;
  L.sc_a = take(n * 32);
  L.sc_b = take((2 * n + 1) * 32);
  L.pts_b = take((2 * n + 1) * sizeof(G1Affine));
  L.ypart = take(blocks * 32);
  L.ticket = take(4);
  L.msm_a = take(var_msm_scratch_bytes(n));
  L.msm_b = take(var_msm_scratch_bytes(2 * n + 1));
  L.total = off;
  return L;
}
size_t batch_partials_scratch_bytes(int n_local) { return rlc_layout((size_t)std::max(n_local, 1)).total; }
// st2 / ev_fork / ev_join: the two MSMs run side by side (the small one on st2)
void launch_batch_partials(void* d_partial288, const void* d_r, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y,
                           size_t first, int n_local, void* d_scratch, cudaStream_t st, cudaStream_t st2, cudaEvent_t ev_fork, cudaEvent_t ev_join) {
  const size_t n = (size_t)std::max(n_local, 0);
  const RlcLayout L = rlc_layout(std::max<size_t>(n, 1));
  uint8_t* base = (uint8_t*)d_scratch;
  uint8_t* out = (uint8_t*)d_partial288;
  cudaMemsetAsync(base + L.ticket, 0, 4, st);
  cudaMemsetAsync(out + 96, 0, 96, st);   // proof_z_lincomb travels inside the third point
  if (n == 0) {
    cudaMemsetAsync(out, 0, 288, st);
    return;
  }
  const int blocks = (int)((n + RLC_THREADS - 1) / RLC_THREADS);
  rlc_scalars_kernel<<<blocks, RLC_THREADS, 0, st>>>((uint32_t*)(base + L.sc_a), (uint32_t*)(base + L.sc_b), (G1Affine*)(base + L.pts_b),
                                                     (uint32_t*)(base + L.ypart), (uint32_t*)(base + L.ticket), (const uint32_t*)d_r,
                                                     (const G1Affine*)d_c_aff, (const G1Affine*)d_pi_aff, (const uint32_t*)d_z, (const uint32_t*)d_y,
                                                     (unsigned long long)first, (int)n);
  count_launch();
  cudaEventRecord(ev_fork, st);
  cudaStreamWaitEvent(st2, ev_fork, 0);
  launch_var_msm_mont(out, d_pi_aff, base + L.sc_a, n, base + L.msm_a, st2);
  cudaEventRecord(ev_join, st2);
  launch_var_msm_mont(out + 192, base + L.pts_b, base + L.sc_b, 2 * n + 1, base + L.msm_b, st);
  cudaStreamWaitEvent(st, ev_join, 0);
}
void launch_batch_final(int* d_ok, const void* d_partials288, int n_ranks, const void* d_prep0, const void* d_prep1, cudaStream_t st) {
  batch_final_kernel<<<1, LW_PAIR_LANES, 0, st>>>(d_ok, (const uint8_t*)d_partials288, n_ranks, (const G2Prepared*)d_prep0, (const G2Prepared*)d_prep1, 0);
  count_launch();
}
void launch_batch_final_each(int* d_ok, const void* d_partials288, int n_checks, const void* d_prep0, const void* d_prep1, cudaStream_t st) {
  if (n_checks <= 0) return;
  batch_final_kernel<<<n_checks, LW_PAIR_LANES, 0, st>>>(d_ok, (const uint8_t*)d_partials288, 1, (const G2Prepared*)d_prep0, (const G2Prepared*)d_prep1, 0);
  count_launch();
}
void launch_batch_final_chain(int* d_ok, const void* d_partials288, int n_checks, const void* d_preps, cudaStream_t st) {
  if (n_checks <= 0) return;
  const G2Prepared* p = (const G2Prepared*)d_preps;
  batch_final_kernel<<<n_checks, LW_PAIR_LANES, 0, st>>>(d_ok, (const uint8_t*)d_partials288, 1, p, p + 1, 1);
  count_launch();
}
}  // namespace lw
