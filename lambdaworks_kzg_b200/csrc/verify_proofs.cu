// Many independent single-opening checks (lwkzg_verify_kzg_proofs): for every item
//        e(C - y G + z pi, g2_0) * e(-pi, g2_1) == 1,
// verify_single_kernel's equation (verify.cu), built for throughput instead of latency.  verify_single_kernel runs
// its ladders on one lane of each warp and its pairing on a 64-lane group; here every item is one THREAD in both
// stages, so all 32 lanes of a warp issue the same multiplications for 32 different items.
//
// The decoding before these kernels (codec.cu, le.cu, poly.cu) runs the r-torsion tests inside the decompression:
// at throughput they are thread-per-point work like the rest of the decompression, and the G1 stage below may then
// use the GLV endomorphism on C and pi unconditionally -- a rejected point arrives as infinity, a rejected scalar as 0.
#include "kernels.h"
#include "pairing.cuh"

namespace lw {

// ---- G1 stage: P = C + [y](-G) + [z] pi and -pi, one item per thread.
// With the GLV split k = q x^2 + m (m, q < 2^128) and phi'(B) = (beta x_B, -y_B) = [x^2]B on the r-torsion, the four
// 128-bit scalars ym, yq, zm, zq act on the bases -G, phi'(-G), pi, phi'(pi).  The ladder is joint over the four
// (Straus): one doubling and ONE addition of a 16-entry table of subset sums per bit.  Every lane runs the same
// schedule -- 128 doublings, 128 table additions -- whatever its scalars, so a warp never executes an addition on
// behalf of a few of its lanes (a separate conditional addition per scalar bit costs the warp 4 additions per bit).
// glv_g == 0 (a mode-0 setup whose g1[0] is not in G1, where phi' is not [x^2]): y acts on -G as one 256-bit scalar
// and the ladder runs 256 bits; the same for every lane of the launch.
constexpr int VP_G1_THREADS = 128;
__global__ void __launch_bounds__(VP_G1_THREADS) verify_proofs_g1_kernel(G1Affine* __restrict__ pts, const G1Affine* __restrict__ c_aff,
                                                                         const G1Affine* __restrict__ pi_aff, const uint32_t* __restrict__ z,
                                                                         const uint32_t* __restrict__ y, const G1Affine* __restrict__ g_in, int glv_g, int n) {
  const int i = blockIdx.x * VP_G1_THREADS + threadIdx.x;
  if (i >= n) return;
  const G1Affine C = c_aff[i], PI = pi_aff[i];
  uint32_t yk[8], zk[8], s[4][8];
  for (int w = 0; w < 8; w++) { yk[w] = y[(size_t)i * 8 + w]; zk[w] = z[(size_t)i * 8 + w]; }
  for (int j = 0; j < 4; j++)
    for (int w = 0; w < 8; w++) s[j][w] = 0;
  Fp beta;
  for (int w = 0; w < 12; w++) beta.l[w] = k::FP_BETA[w];
  G1Affine b[4];
  b[0] = g1a_neg(*g_in);
  b[1] = g1a_inf();
  if (glv_g) {
    glv_split(s[1], s[0], yk);
    b[1].x = fp_mul(b[0].x, beta);   // phi'(-G) = (beta x_G, y_G); infinity (0, 0) stays infinity
    b[1].y = g_in->y;
  } else {
    for (int w = 0; w < 8; w++) s[0][w] = yk[w];
  }
  glv_split(s[3], s[2], zk);
  b[2] = PI;
  b[3].x = fp_mul(PI.x, beta);
  b[3].y = fp_neg(PI.y);
  G1Xyzz t[16];
  t[0] = xyzz_inf();
  for (int m = 1; m < 16; m++) {
    const int j = __ffs(m) - 1;
    t[m] = t[m & (m - 1)];
    xyzz_madd_ni(t[m], b[j]);
  }
  G1Xyzz acc = xyzz_inf();
  const int nbits = glv_g ? 128 : 256;
  for (int bit = nbits - 1; bit >= 0; bit--) {
    xyzz_dbl_ni(acc);
    const int w = bit >> 5, sh = bit & 31;
    const int m = ((s[0][w] >> sh) & 1) | (((s[1][w] >> sh) & 1) << 1) | (((s[2][w] >> sh) & 1) << 2) | (((s[3][w] >> sh) & 1) << 3);
    xyzz_add_ni(acc, t[m]);
  }
  xyzz_madd_ni(acc, C);
  pts[2 * (size_t)i] = xyzz_to_affine(acc);
  pts[2 * (size_t)i + 1] = g1a_neg(PI);
}

// ---- pairing stage, one item per thread: the single-thread Miller loop of pairing.cuh over the two fixed prepared
// G2 points, then its final exponentiation.  A term whose G1 point is infinity contributes 1 and is skipped by that
// lane alone.  ok[i] = status[i] == 0 && product == 1.
// Timed against one 64-lane group per item on the pairing_warp.cuh phases (one group per 64-thread block, the layout
// of batch_final_kernel), device-resident on a B200: 1024 items 30.1 vs 14.6 ms, 16384 items 32.4 vs 108.2 ms
// (profiles/r03_verify_proofs_bench_b200.jsonl).  The group layout wins only while the GPU is mostly idle; this call
// exists for many items, and a single opening is faster through verify_kzg_proof either way.
constexpr int VP_PAIR_THREADS = 64;
__global__ void __launch_bounds__(VP_PAIR_THREADS) verify_proofs_pairing_kernel(int* __restrict__ ok, const int* __restrict__ status,
                                                                                const G1Affine* __restrict__ pts, const G2Prepared* __restrict__ prep0,
                                                                                const G2Prepared* __restrict__ prep1, int n) {
  const int i = blockIdx.x * VP_PAIR_THREADS + threadIdx.x;
  if (i >= n) return;
  const G1Affine p0 = pts[2 * (size_t)i], p1 = pts[2 * (size_t)i + 1];
  const bool use0 = !g1a_is_inf(p0) && !prep0->infinity, use1 = !g1a_is_inf(p1) && !prep1->infinity;
  Fp12 f = fp12_one();
  int step = 0;
  for (int bit = 62; bit >= 0; bit--) {
    f = fp12_sqr(f);
    if (use0) f = line_mul(f, prep0->line[step], p0);
    if (use1) f = line_mul(f, prep1->line[step], p1);
    step++;
    if ((k::BLS_X_ABS >> bit) & 1ull) {
      if (use0) f = line_mul(f, prep0->line[step], p0);
      if (use1) f = line_mul(f, prep1->line[step], p1);
      step++;
    }
  }
  const bool one = fp12_is_one(final_exponentiation(fp12_conj(f)));   // conj: x < 0
  ok[i] = (status[i] == 0 && one) ? 1 : 0;
}

void launch_verify_proofs_g1(void* d_pts, const void* d_c_aff, const void* d_pi_aff, const void* d_z, const void* d_y, const void* d_g_aff, bool glv_g, int n,
                             cudaStream_t st) {
  if (n <= 0) return;
  verify_proofs_g1_kernel<<<(n + VP_G1_THREADS - 1) / VP_G1_THREADS, VP_G1_THREADS, 0, st>>>(
      (G1Affine*)d_pts, (const G1Affine*)d_c_aff, (const G1Affine*)d_pi_aff, (const uint32_t*)d_z, (const uint32_t*)d_y, (const G1Affine*)d_g_aff,
      glv_g ? 1 : 0, n);
  count_launch();
}
void launch_verify_proofs_pairing(int* d_ok, const int* d_status, const void* d_pts, const void* d_prep0, const void* d_prep1, int n, cudaStream_t st) {
  if (n <= 0) return;
  verify_proofs_pairing_kernel<<<(n + VP_PAIR_THREADS - 1) / VP_PAIR_THREADS, VP_PAIR_THREADS, 0, st>>>(
      d_ok, d_status, (const G1Affine*)d_pts, (const G2Prepared*)d_prep0, (const G2Prepared*)d_prep1, n);
  count_launch();
}

}  // namespace lw
