// Trusted-setup decoding on the device (load_trusted_setup[_file],
// /root/reference/src/lib.rs:709-802, src/srs.rs:25-128): every compressed
// point is validated exactly like the reference's loaders do (G1: curve +
// subgroup; G2: curve only) and returned as canonical integers so the host can
// lay out KZGSettings.g1_values / g2_values the way src/srs.rs:131-213 does.
// The c-kzg-4844 loaders decode G2 strictly (subgroup included) and derive the
// weights of their setup check (lwkzg.cu, settings_from_ckzg) here.
#include "fp2.cuh"
#include "g1.cuh"
#include "kernels_setup.h"
#include "sha256.cuh"

namespace lw {

__global__ void __launch_bounds__(32) setup_decode_g1_kernel(uint32_t* __restrict__ canon24, int* __restrict__ status, const uint8_t* __restrict__ in48, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t buf[48];
  for (int k = 0; k < 48; k++) buf[k] = in48[(size_t)i * 48 + k];
  G1Affine p;
  bool ok = g1_decompress(p, buf);
  status[i] = ok ? 0 : 2;
  Fp x = fp_zero(), y = fp_zero();
  if (ok && !g1a_is_inf(p)) { x = fp_from_mont(p.x); y = fp_from_mont(p.y); }
  for (int k = 0; k < 12; k++) { canon24[i * 24 + k] = x.l[k]; canon24[i * 24 + 12 + k] = y.l[k]; }
}

// out: x.c0, x.c1, y.c0, y.c1 canonical (48 u32); status 0 ok, 1 = infinity, 2 = rejected
__global__ void __launch_bounds__(32) setup_decode_g2_kernel(uint32_t* __restrict__ canon48, int* __restrict__ status, const uint8_t* __restrict__ in96, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t buf[96];
  for (int k = 0; k < 96; k++) buf[k] = in96[(size_t)i * 96 + k];
  G2Affine q;
  bool inf = false;
  bool ok = g2_decompress(q, inf, buf);
  status[i] = ok ? (inf ? 1 : 0) : 2;
  Fp c[4] = {fp_zero(), fp_zero(), fp_zero(), fp_zero()};
  if (ok && !inf) { c[0] = fp_from_mont(q.x.c0); c[1] = fp_from_mont(q.x.c1); c[2] = fp_from_mont(q.y.c0); c[3] = fp_from_mont(q.y.c1); }
  for (int j = 0; j < 4; j++)
    for (int k = 0; k < 12; k++) canon48[i * 48 + j * 12 + k] = c[j].l[k];
}

// ------------------------------------------------------------------ c-kzg-4844 setups (lwkzg_load_trusted_setup_ckzg)
// Jacobian coordinates on the twist y^2 = x^3 + 4 (1 + u); z = 0 is the point at infinity
struct G2Jac {
  Fp2 x, y, z;
};
// dbl-2009-l (a = 0)
LW_COLD void g2j_dbl(G2Jac& p) {
  const Fp2 a = fp2_sqr(p.x), b = fp2_sqr(p.y), c = fp2_sqr(b);
  const Fp2 d = fp2_dbl(fp2_sub(fp2_sub(fp2_sqr(fp2_add(p.x, b)), a), c));
  const Fp2 e = fp2_add(fp2_dbl(a), a);
  const Fp2 z3 = fp2_dbl(fp2_mul(p.y, p.z));
  p.x = fp2_sub(fp2_sqr(e), fp2_dbl(d));
  p.y = fp2_sub(fp2_mul(e, fp2_sub(d, p.x)), fp2_dbl(fp2_dbl(fp2_dbl(c))));
  p.z = z3;
}
// p += q, q affine and finite (madd-2007-bl); complete: p at infinity, p == q and p == -q are handled
LW_COLD void g2j_madd(G2Jac& p, const G2Affine& q) {
  if (fp2_is_zero(p.z)) { p.x = q.x; p.y = q.y; p.z = fp2_one(); return; }
  const Fp2 z1z1 = fp2_sqr(p.z);
  const Fp2 h = fp2_sub(fp2_mul(q.x, z1z1), p.x);
  const Fp2 r = fp2_dbl(fp2_sub(fp2_mul(q.y, fp2_mul(p.z, z1z1)), p.y));
  if (fp2_is_zero(h)) {
    if (fp2_is_zero(r)) g2j_dbl(p);
    else p.z = fp2_zero();
    return;
  }
  const Fp2 hh = fp2_sqr(h);
  const Fp2 i = fp2_dbl(fp2_dbl(hh));
  const Fp2 j = fp2_mul(h, i);
  const Fp2 v = fp2_mul(p.x, i);
  const Fp2 x3 = fp2_sub(fp2_sub(fp2_sqr(r), j), fp2_dbl(v));
  const Fp2 y3 = fp2_sub(fp2_mul(r, fp2_sub(v, x3)), fp2_dbl(fp2_mul(p.y, j)));
  p.z = fp2_sub(fp2_sub(fp2_sqr(fp2_add(p.z, h)), z1z1), hh);
  p.x = x3;
  p.y = y3;
}
// [r]Q == O for a finite Q on the twist: Q is in G2 (blst's subgroup test decides the same set)
LW_COLD bool g2_in_subgroup(const G2Affine& q) {
  G2Jac acc;
  acc.x = q.x; acc.y = q.y; acc.z = fp2_one();
  for (int bit = 253; bit >= 0; bit--) {   // r < 2^255, bit 254 set: acc starts at [1]Q
    g2j_dbl(acc);
    if ((k::FR_MOD[bit >> 5] >> (bit & 31)) & 1u) g2j_madd(acc, q);
  }
  return fp2_is_zero(acc.z);
}

// blst-strict G2 decoding: compression flag set, no infinity (a setup point never is one), both x coordinates
// canonical (< p), on the twist, in G2.  status: 0 ok, 1 encoding, 2 not on the twist, 3 not in G2
__global__ void __launch_bounds__(32) setup_decode_g2_strict_kernel(uint32_t* __restrict__ canon48, int* __restrict__ status,
                                                                   const uint8_t* __restrict__ in96, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t buf[96];
  for (int k = 0; k < 96; k++) buf[k] = in96[(size_t)i * 96 + k];
  int code = 0;
  if ((buf[0] & 0xC0) != 0x80) {
    code = 1;
  } else {
    Fp c1, c0;
    for (int k = 0; k < 12; k++) {
      const uint8_t* q1 = buf + 44 - 4 * k;
      const uint8_t* q0 = buf + 92 - 4 * k;
      c1.l[k] = ((uint32_t)q1[0] << 24) | ((uint32_t)q1[1] << 16) | ((uint32_t)q1[2] << 8) | (uint32_t)q1[3];
      c0.l[k] = ((uint32_t)q0[0] << 24) | ((uint32_t)q0[1] << 16) | ((uint32_t)q0[2] << 8) | (uint32_t)q0[3];
    }
    c1.l[11] &= 0x1FFFFFFFu;
    if (!limbs_lt<12>(c1.l, k::FP_MOD) || !limbs_lt<12>(c0.l, k::FP_MOD)) code = 1;
  }
  G2Affine q;
  bool inf = false;
  if (code == 0 && !g2_decompress(q, inf, buf)) code = 2;
  if (code == 0 && !g2_in_subgroup(q)) code = 3;
  status[i] = code;
  Fp c[4] = {fp_zero(), fp_zero(), fp_zero(), fp_zero()};
  if (code == 0) { c[0] = fp_from_mont(q.x.c0); c[1] = fp_from_mont(q.x.c1); c[2] = fp_from_mont(q.y.c0); c[3] = fp_from_mont(q.y.c1); }
  for (int j = 0; j < 4; j++)
    for (int k = 0; k < 12; k++) canon48[i * 48 + j * 12 + k] = c[j].l[k];
}

// rho = SHA-256(msg) read big-endian, mod r (canonical).  msg: nblocks 64-byte blocks, padding included.  One warp.
__global__ void __launch_bounds__(32) setup_rho_kernel(uint32_t* __restrict__ rho, const uint32_t* __restrict__ msg, int nblocks) {
  __shared__ uint32_t wk[64 * 32];
  Sha256State s;
  sha256_init(s);
  sha256_warp_blocks(s, nblocks, [&](int blk, uint32_t* w) {
    for (int i = 0; i < 16; i++) w[i] = bswap32(msg[(size_t)blk * 16 + i]);
  }, wk);
  if (threadIdx.x != 0) return;
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = s.h[7 - i];
  mod_reduce_small<FrCfg, 2>(r.l);
  for (int i = 0; i < 8; i++) rho[i] = r.l[i];
}

// k < 4096: sc[k] = rho^k (canonical) and blob[brp(k)] = rho^k (32 bytes big-endian), i.e. the MODE_DENEB blob whose
// polynomial takes the value rho^k at w^k
__global__ void setup_rho_powers_kernel(uint32_t* __restrict__ sc, uint8_t* __restrict__ blob, const uint32_t* __restrict__ rho) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= N_POINTS) return;
  Fr base;
  for (int i = 0; i < 8; i++) base.l[i] = rho[i];
  base = fr_to_mont(base);
  Fr acc = fr_one();
  for (int bit = 11; bit >= 0; bit--) {
    acc = fr_sqr(acc);
    if ((k >> bit) & 1u) acc = fr_mul(acc, base);
  }
  acc = fr_from_mont(acc);
  for (int i = 0; i < 8; i++) sc[k * 8 + i] = acc.l[i];
  fr_canon_to_be32(blob + (size_t)(__brev(k) >> 20) * 32, acc);
}

// sc[j] = -coef[j] (canonical; coef in Montgomery form)
__global__ void setup_neg_coef_kernel(uint32_t* __restrict__ sc, const Fr* __restrict__ coef) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N_POINTS) return;
  const Fr v = fr_from_mont(fr_neg(coef[j]));
  for (int i = 0; i < 8; i++) sc[j * 8 + i] = v.l[i];
}

void launch_setup_decode_g1(void* d_canon24, int* d_status, const void* d_in48, int n, cudaStream_t st) {
  if (n <= 0) return;
  setup_decode_g1_kernel<<<(n + 31) / 32, 32, 0, st>>>((uint32_t*)d_canon24, d_status, (const uint8_t*)d_in48, n);
  count_launch();
}
void launch_setup_decode_g2(void* d_canon48, int* d_status, const void* d_in96, int n, cudaStream_t st) {
  if (n <= 0) return;
  setup_decode_g2_kernel<<<(n + 31) / 32, 32, 0, st>>>((uint32_t*)d_canon48, d_status, (const uint8_t*)d_in96, n);
  count_launch();
}

void launch_setup_decode_g2_strict(void* d_canon48, int* d_status, const void* d_in96, int n, cudaStream_t st) {
  if (n <= 0) return;
  setup_decode_g2_strict_kernel<<<(n + 31) / 32, 32, 0, st>>>((uint32_t*)d_canon48, d_status, (const uint8_t*)d_in96, n);
  count_launch();
}
void launch_setup_rho(void* d_rho, const void* d_msg, int nblocks, cudaStream_t st) {
  setup_rho_kernel<<<1, 32, 0, st>>>((uint32_t*)d_rho, (const uint32_t*)d_msg, nblocks);
  count_launch();
}
void launch_setup_rho_powers(void* d_sc, void* d_blob, const void* d_rho, cudaStream_t st) {
  setup_rho_powers_kernel<<<N_POINTS / 128, 128, 0, st>>>((uint32_t*)d_sc, (uint8_t*)d_blob, (const uint32_t*)d_rho);
  count_launch();
}
void launch_setup_neg_coef(void* d_sc, const void* d_coef, cudaStream_t st) {
  setup_neg_coef_kernel<<<N_POINTS / 128, 128, 0, st>>>((uint32_t*)d_sc, (const Fr*)d_coef);
  count_launch();
}

}  // namespace lw
