// Device-math harness: the math headers of the library, one operation per kernel, one case per thread.
//
// Built twice from this one source (tests/_device_math.py):
//   * nvcc for sm_100a with the library's flags -- the headers run on the device, in warps whose lanes take
//     different branches of the same operation (the layouts are chosen by the caller through the case order,
//     the block size and odd_lanes_only);
//   * g++ -x c++ -DLWKZG_HOST_EMUL -- the same per-case functions in a host loop over the cases.  Pieces that
//     only exist on the device (warp-cooperative SHA-256, the pairing on real lanes, the MSM helpers of
//     msm_common.cuh) are not compiled there and report DM_UNSUPPORTED.
//
// Records are little-endian u32 words.  Field elements are their 12 (Fp) or 8 (Fr) limbs exactly as the device
// holds them (Montgomery form unless the operation says otherwise), points are G1Affine / G1Xyzz / Fp2 structs
// word for word, byte strings are packed four bytes to a word in memory order.  The layout of each operation's
// input and output record is given next to its id below and mirrored in tests/test_device_math.py.
#include <stdint.h>
#include <stddef.h>
#include <string.h>

#include "../../lambdaworks_kzg_b200/csrc/g1.cuh"
#include "../../lambdaworks_kzg_b200/csrc/fpinv.cuh"
#include "../../lambdaworks_kzg_b200/csrc/fp2.cuh"
#include "../../lambdaworks_kzg_b200/csrc/sha256.cuh"
#include "../../lambdaworks_kzg_b200/csrc/recode.cuh"
#include "../../lambdaworks_kzg_b200/csrc/lepoly.cuh"
#if !defined(LWKZG_HOST_EMUL)
#include "../../lambdaworks_kzg_b200/csrc/msm_ba.cuh"
#include "../../lambdaworks_kzg_b200/csrc/pairing_warp.cuh"
#endif

using namespace lw;

enum : int {
  DM_UNSUPPORTED = -1,
  DM_BAD_ARGS = -2,
};

// Operation ids (in -> out, in words).
enum : int {
  OP_FP_ARITH = 0,          // a[12] b[12] -> add sub neg dbl mul mul_nv sqr sqr_nv to_mont(a) from_mont(a), 10 x 12
  OP_FR_ARITH = 1,          // a[8] b[8] -> add sub neg dbl mul sqr to_mont(a) from_mont(a), 8 x 8
  OP_FP_FROM_BE48 = 2,      // 48 bytes (top 3 bits clear) -> fp_from_be48 [12]
  OP_FR_FROM_BE = 3,        // 32 bytes -> fr_canon_from_be32 [8], fr_canon_from_be_words [8]
  OP_FP_INV_GCD = 4,        // a[12] -> [12]
  OP_FP_INV_FERMAT = 5,     // a[12] -> [12]
  OP_FR_INV = 6,            // a[8] -> [8]
  OP_FR_BATCH_INV = 7,      // cnt, d[32][8] -> inv[32][8]
  OP_FR_ZN_MINUS_ONE = 8,   // z[8] -> [8]
  // group law: in = A (G1Xyzz, 48) | B (G1Affine, 24) | Bx (G1Xyzz, 48)
  OP_XYZZ_MADD = 10,        // A += B           -> G1Xyzz
  OP_XYZZ_MADD_HOT = 11,
  OP_XYZZ_MADD_NI = 12,
  OP_XYZZ_MADD_RARE = 13,
  OP_XYZZ_ADD = 14,         // A += Bx          -> G1Xyzz
  OP_XYZZ_ADD_NI = 15,
  OP_XYZZ_DBL = 16,         // 2 A              -> G1Xyzz
  OP_XYZZ_DBL_NI = 17,
  OP_XYZZ_DBL_AFFINE = 18,  // 2 B              -> G1Xyzz
  OP_G1A_DBL_NI = 19,       // 2 B              -> G1Affine (device only: msm_ba.cuh)
  OP_XYZZ_TO_AFFINE = 20,   // A                -> G1Affine
  OP_XYZZ_EQ = 21,          // A == Bx          -> [1]
  // scalars: in = base (G1Affine, 24) | k[8] | c
  OP_G1_MUL = 30,           // -> g1_mul_scalar (48) | g1_mul_scalar_glv (48)
  OP_GLV_RECODE = 31,       // -> glv_split q[4] m[4] | glv_split_barrett q[4] m[4] | digits of m[W] | of q[W] (W <= 16)
  // codecs
  OP_G1_COMPRESS = 40,      // G1Affine -> 48 bytes
  OP_G1_DECOMPRESS = 41,    // 48 bytes -> ok | G1Affine  (lax, subgroup check)
  OP_G1_DECOMPRESS_NOSUB = 42,  //                        (lax, no subgroup check)
  OP_G1_DECOMPRESS_STRICT = 43, //                        (strict, subgroup check)
  OP_G1_CHECKS = 44,        // G1Affine -> on_curve | in_subgroup
  OP_G2_DECOMPRESS = 45,    // 96 bytes -> status (0 reject, 1 point, 2 infinity) | G2Affine (48)
  OP_FP2_INV = 46,          // Fp2 (24) -> Fp2
  OP_FP2_SQRT = 47,         // Fp2 (24) -> ok | Fp2
  // hashing
  OP_SHA256_ONESHOT = 50,   // len | message bytes -> 32 bytes
  OP_SHA256_WARP = 51,      // one warp per case: nblocks | pre-padded blocks -> 32 bytes (device only)
  // pairing, one LW_PAIR_LANES block per case: P0 P1 (G1Affine) | Q0 Q1 (G2Affine) ->
  //   warp_pairing_product Fp12 (144) | single-thread final_exponentiation(miller_loop) Fp12 (144) |
  //   warp_fp12_is_one | pairing_product_is_one  (device only)
  OP_PAIRING = 60,
};

constexpr int FR_BATCH_MAX = LE_INV_GROUP;

template <class T>
LW_INL void ld(T& v, const uint32_t* w) {
  uint32_t* d = reinterpret_cast<uint32_t*>(&v);
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) d[i] = w[i];
}
template <class T>
LW_INL void st(uint32_t* w, const T& v) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(&v);
  for (int i = 0; i < (int)(sizeof(T) / 4); i++) w[i] = s[i];
}

template <int OP>
LW_INL void run_case(const uint32_t* in, uint32_t* out) {
  if constexpr (OP == OP_FP_ARITH) {
    Fp a, b;
    ld(a, in); ld(b, in + 12);
    st(out + 0, fp_add(a, b));
    st(out + 12, fp_sub(a, b));
    st(out + 24, fp_neg(a));
    st(out + 36, fp_dbl(a));
    st(out + 48, fp_mul(a, b));
    st(out + 60, fp_mul_nv(a, b));
    st(out + 72, fp_sqr(a));
    st(out + 84, fp_sqr_nv(a));
    st(out + 96, fp_to_mont(a));
    st(out + 108, fp_from_mont(a));
  } else if constexpr (OP == OP_FR_ARITH) {
    Fr a, b;
    ld(a, in); ld(b, in + 8);
    st(out + 0, fr_add(a, b));
    st(out + 8, fr_sub(a, b));
    st(out + 16, fr_neg(a));
    Fr d; mod_dbl<FrCfg>(d.l, a.l);
    st(out + 24, d);
    st(out + 32, fr_mul(a, b));
    st(out + 40, fr_sqr(a));
    st(out + 48, fr_to_mont(a));
    st(out + 56, fr_from_mont(a));
  } else if constexpr (OP == OP_FP_FROM_BE48) {
    st(out, fp_from_be48(reinterpret_cast<const uint8_t*>(in)));
  } else if constexpr (OP == OP_FR_FROM_BE) {
    st(out, fr_canon_from_be32(reinterpret_cast<const uint8_t*>(in)));
    st(out + 8, fr_canon_from_be_words(in));
  } else if constexpr (OP == OP_FP_INV_GCD) {
    Fp a; ld(a, in);
    st(out, fp_inv_gcd(a));
  } else if constexpr (OP == OP_FP_INV_FERMAT) {
    Fp a; ld(a, in);
    st(out, fp_inv_fermat(a));
  } else if constexpr (OP == OP_FR_INV) {
    Fr a; ld(a, in);
    st(out, fr_inv(a));
  } else if constexpr (OP == OP_FR_BATCH_INV) {
    int cnt = (int)in[0];
    cnt = cnt < 0 ? 0 : (cnt > FR_BATCH_MAX ? FR_BATCH_MAX : cnt);
    Fr d[FR_BATCH_MAX], inv[FR_BATCH_MAX];
    for (int k = 0; k < FR_BATCH_MAX; k++) { ld(d[k], in + 1 + 8 * k); inv[k] = fr_zero(); }
    fr_batch_inv_group(inv, d, cnt);
    for (int k = 0; k < FR_BATCH_MAX; k++) st(out + 8 * k, inv[k]);
  } else if constexpr (OP == OP_FR_ZN_MINUS_ONE) {
    Fr z; ld(z, in);
    st(out, fr_zn_minus_one(z));
  } else if constexpr (OP >= OP_XYZZ_MADD && OP <= OP_XYZZ_EQ) {
    G1Xyzz A, Bx;
    G1Affine B;
    ld(A, in); ld(B, in + 48); ld(Bx, in + 72);
    if constexpr (OP == OP_XYZZ_MADD) { xyzz_madd(A, B); st(out, A); }
    if constexpr (OP == OP_XYZZ_MADD_HOT) { xyzz_madd_hot(A, B); st(out, A); }
    if constexpr (OP == OP_XYZZ_MADD_NI) { xyzz_madd_ni(A, B); st(out, A); }
    if constexpr (OP == OP_XYZZ_MADD_RARE) { xyzz_madd_rare(A, B); st(out, A); }
    if constexpr (OP == OP_XYZZ_ADD) { xyzz_add(A, Bx); st(out, A); }
    if constexpr (OP == OP_XYZZ_ADD_NI) { xyzz_add_ni(A, Bx); st(out, A); }
    if constexpr (OP == OP_XYZZ_DBL) st(out, xyzz_dbl(A));
    if constexpr (OP == OP_XYZZ_DBL_NI) { xyzz_dbl_ni(A); st(out, A); }
    if constexpr (OP == OP_XYZZ_DBL_AFFINE) st(out, xyzz_dbl_affine(B));
#if !defined(LWKZG_HOST_EMUL)
    if constexpr (OP == OP_G1A_DBL_NI) st(out, g1a_dbl_ni(B));
#endif
    if constexpr (OP == OP_XYZZ_TO_AFFINE) st(out, xyzz_to_affine(A));
    if constexpr (OP == OP_XYZZ_EQ) out[0] = xyzz_eq(A, Bx) ? 1u : 0u;
  } else if constexpr (OP == OP_G1_MUL) {
    G1Affine p; ld(p, in);
    st(out, g1_mul_scalar(p, in + 24, 8));
    st(out + 48, g1_mul_scalar_glv(p, in + 24));
  } else if constexpr (OP == OP_GLV_RECODE) {
    const uint32_t* k8 = in + 24;
    const int c = (int)in[32];
    glv_split(out, out + 4, k8);
    uint32_t q[4], m[4];
    glv_split_barrett(q, m, k8);
    for (int i = 0; i < 4; i++) { out[8 + i] = q[i]; out[12 + i] = m[i]; }
    const int W = glv_num_windows(c);
    for (int h = 0; h < 2; h++) {
      const uint32_t* v = h ? q : m;
      int carry = 0;
      for (int j = 0; j < W; j++) out[16 + 16 * h + j] = (uint32_t)glv_digit([&](int w) { return v[w]; }, c, W, j, carry);
    }
  } else if constexpr (OP == OP_G1_COMPRESS) {
    G1Affine p; ld(p, in);
    g1_compress(reinterpret_cast<uint8_t*>(out), p);
  } else if constexpr (OP == OP_G1_DECOMPRESS || OP == OP_G1_DECOMPRESS_NOSUB || OP == OP_G1_DECOMPRESS_STRICT) {
    G1Affine p = g1a_inf();
    const uint8_t* b = reinterpret_cast<const uint8_t*>(in);
    bool ok;
    if constexpr (OP == OP_G1_DECOMPRESS) ok = g1_decompress(p, b, true);
    else if constexpr (OP == OP_G1_DECOMPRESS_NOSUB) ok = g1_decompress(p, b, false);
    else ok = g1_decompress_strict(p, b, true);
    out[0] = ok ? 1u : 0u;
    st(out + 1, ok ? p : g1a_inf());
  } else if constexpr (OP == OP_G1_CHECKS) {
    G1Affine p; ld(p, in);
    out[0] = g1a_on_curve(p) ? 1u : 0u;
    out[1] = g1_in_subgroup(p) ? 1u : 0u;
  } else if constexpr (OP == OP_G2_DECOMPRESS) {
    G2Affine q;
    bool inf = false;
    const bool ok = g2_decompress(q, inf, reinterpret_cast<const uint8_t*>(in));
    out[0] = !ok ? 0u : (inf ? 2u : 1u);
    if (!ok) { q.x = fp2_zero(); q.y = fp2_zero(); }
    st(out + 1, q);
  } else if constexpr (OP == OP_FP2_INV) {
    Fp2 a; ld(a, in);
    st(out, fp2_inv(a));
  } else if constexpr (OP == OP_FP2_SQRT) {
    Fp2 a, r = fp2_zero(); ld(a, in);
    const bool ok = fp2_sqrt(r, a);
    out[0] = ok ? 1u : 0u;
    st(out + 1, ok ? r : fp2_zero());
  } else if constexpr (OP == OP_SHA256_ONESHOT) {
    uint8_t d[32];
    sha256_oneshot(d, reinterpret_cast<const uint8_t*>(in + 1), (size_t)in[0]);
    for (int i = 0; i < 32; i++) reinterpret_cast<uint8_t*>(out)[i] = d[i];
  }
}

#if !defined(LWKZG_HOST_EMUL)
// ---------------------------------------------------------------- device backend
// Thread t runs case t; with odd_lanes_only, thread t runs case t / 2 when t is odd and even threads branch
// around the call (a caller whose warp is split in two).
template <int OP>
__global__ void dm_kernel(int n, int odd_lanes_only, const uint8_t* __restrict__ in, size_t in_stride, uint8_t* __restrict__ out,
                          size_t out_stride) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i = odd_lanes_only ? (t >> 1) : t;
  if (odd_lanes_only && !(t & 1)) return;
  if (i >= n) return;
  run_case<OP>(reinterpret_cast<const uint32_t*>(in + (size_t)i * in_stride), reinterpret_cast<uint32_t*>(out + (size_t)i * out_stride));
}

// one warp per case: nblocks | blocks (16 big-endian words each, stored as bytes)
__global__ void __launch_bounds__(32) dm_sha256_warp_kernel(const uint8_t* __restrict__ in, size_t in_stride, uint8_t* __restrict__ out,
                                                             size_t out_stride) {
  __shared__ uint32_t wk[64 * 32];
  const uint32_t* rec = reinterpret_cast<const uint32_t*>(in + (size_t)blockIdx.x * in_stride);
  const int nblocks = (int)rec[0];
  Sha256State s;
  sha256_init(s);
  sha256_warp_blocks(s, nblocks, [&](int blk, uint32_t* w) {
    for (int i = 0; i < 16; i++) w[i] = bswap32(rec[1 + 16 * blk + i]);
  }, wk);
  if (threadIdx.x == 0) sha256_digest_bytes(out + (size_t)blockIdx.x * out_stride, s);
}

__global__ void __launch_bounds__(LW_PAIR_LANES) dm_pairing_kernel(const uint8_t* __restrict__ in, size_t in_stride, uint8_t* __restrict__ out,
                                                                    size_t out_stride) {
  __shared__ WarpPairingMem m;
  __shared__ G2Prepared prep[2];
  __shared__ G1Affine ps[2];
  const uint32_t* rec = reinterpret_cast<const uint32_t*>(in + (size_t)blockIdx.x * in_stride);
  uint32_t* o = reinterpret_cast<uint32_t*>(out + (size_t)blockIdx.x * out_stride);
  if (threadIdx.x < 2) {
    ld(ps[threadIdx.x], rec + 24 * threadIdx.x);
    G2Affine q;
    ld(q, rec + 48 + 48 * threadIdx.x);
    g2_prepare(prep[threadIdx.x], q);
  }
  __syncthreads();
  const G2Prepared* qs[2] = {&prep[0], &prep[1]};
  warp_pairing_product(m, ps, qs, 2);
  if (threadIdx.x == 0) {
    st(o, m.f);
    const G1Affine p2[2] = {ps[0], ps[1]};
    st(o + 144, final_exponentiation(miller_loop(p2, prep, 2)));
    o[288] = warp_fp12_is_one(m.f) ? 1u : 0u;
    o[289] = pairing_product_is_one(p2, prep, 2) ? 1u : 0u;
  }
}

template <int OP>
static cudaError_t launch(int n, int tpb, int odd, const uint8_t* in, size_t in_stride, uint8_t* out, size_t out_stride) {
  const long long threads = odd ? 2ll * n : (long long)n;
  const long long blocks = (threads + tpb - 1) / tpb;
  dm_kernel<OP><<<(unsigned)blocks, tpb>>>(n, odd, in, in_stride, out, out_stride);
  return cudaGetLastError();
}
#endif

#define DM_OPS(X)                                                                                                   \
  X(OP_FP_ARITH) X(OP_FR_ARITH) X(OP_FP_FROM_BE48) X(OP_FR_FROM_BE) X(OP_FP_INV_GCD) X(OP_FP_INV_FERMAT) X(OP_FR_INV) \
  X(OP_FR_BATCH_INV) X(OP_FR_ZN_MINUS_ONE) X(OP_XYZZ_MADD) X(OP_XYZZ_MADD_HOT) X(OP_XYZZ_MADD_NI) X(OP_XYZZ_MADD_RARE) \
  X(OP_XYZZ_ADD) X(OP_XYZZ_ADD_NI) X(OP_XYZZ_DBL) X(OP_XYZZ_DBL_NI) X(OP_XYZZ_DBL_AFFINE) X(OP_XYZZ_TO_AFFINE)        \
  X(OP_XYZZ_EQ) X(OP_G1_MUL) X(OP_GLV_RECODE) X(OP_G1_COMPRESS) X(OP_G1_DECOMPRESS) X(OP_G1_DECOMPRESS_NOSUB)        \
  X(OP_G1_DECOMPRESS_STRICT) X(OP_G1_CHECKS) X(OP_G2_DECOMPRESS) X(OP_FP2_INV) X(OP_FP2_SQRT) X(OP_SHA256_ONESHOT)

extern "C" {

// Runs `n` cases of operation `op`: case i reads in + i * in_stride and writes out + i * out_stride (host
// memory).  Returns 0, the first CUDA error, DM_UNSUPPORTED for an operation this backend does not have, or
// DM_BAD_ARGS.  The device backend allocates, copies, launches and frees within the call.
int dm_run(int op, int n, int threads_per_block, int odd_lanes_only, const void* in, size_t in_stride, void* out, size_t out_stride) {
  if (n < 0 || threads_per_block <= 0 || threads_per_block > 1024) return DM_BAD_ARGS;
  if (n == 0) return 0;
#if defined(LWKZG_HOST_EMUL)
  (void)odd_lanes_only;
  for (int i = 0; i < n; i++) {
    const uint32_t* ci = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(in) + (size_t)i * in_stride);
    uint32_t* co = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(out) + (size_t)i * out_stride);
    switch (op) {
#define DM_CASE(OPID) case OPID: run_case<OPID>(ci, co); break;
      DM_OPS(DM_CASE)
#undef DM_CASE
      default: return DM_UNSUPPORTED;
    }
  }
  return 0;
#else
  uint8_t *din = nullptr, *dout = nullptr;
  cudaError_t e = cudaMalloc(&din, in_stride * (size_t)n);
  if (e == cudaSuccess) e = cudaMalloc(&dout, out_stride * (size_t)n);
  if (e == cudaSuccess) e = cudaMemcpy(din, in, in_stride * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(dout, 0, out_stride * (size_t)n);
  int rc = 0;
  if (e == cudaSuccess) {
    switch (op) {
#define DM_CASE(OPID) case OPID: e = launch<OPID>(n, threads_per_block, odd_lanes_only, din, in_stride, dout, out_stride); break;
      DM_OPS(DM_CASE)
      DM_CASE(OP_G1A_DBL_NI)
#undef DM_CASE
      case OP_SHA256_WARP:
        dm_sha256_warp_kernel<<<n, 32>>>(din, in_stride, dout, out_stride);
        e = cudaGetLastError();
        break;
      case OP_PAIRING:
        dm_pairing_kernel<<<n, LW_PAIR_LANES>>>(din, in_stride, dout, out_stride);
        e = cudaGetLastError();
        break;
      default: rc = DM_UNSUPPORTED;
    }
  }
  if (e == cudaSuccess && rc == 0) e = cudaDeviceSynchronize();
  if (e == cudaSuccess && rc == 0) e = cudaMemcpy(out, dout, out_stride * (size_t)n, cudaMemcpyDeviceToHost);
  const cudaError_t e1 = din ? cudaFree(din) : cudaSuccess;
  const cudaError_t e2 = dout ? cudaFree(dout) : cudaSuccess;
  if (e == cudaSuccess) e = e1 != cudaSuccess ? e1 : e2;
  return e != cudaSuccess ? (int)e : rc;
#endif
}

}  // extern "C"
