// The batch challenge of a batched blob verification (compute_r_powers, utils.rs:156-206), one warp:
//   r = H("RCKZGBATCH___V1_" || le64(4096) || le64(n) || tuples), read big-endian, mod r.
// batch_challenge_kernel (verify.cu) hashes one batch, possibly block range by block range; the per-batch kernel of
// lwkzg_verify_blob_kzg_proof_batches (verify_batches.cu) hashes one whole batch per warp.
#pragma once
#include "field.cuh"
#include "sha256.cuh"

namespace lw {

constexpr int BCH_INIT = 1, BCH_FINAL = 2, BCH_LE = 4, BCH_BE_HDR = 8;

// wire: 0 = reference, 1 = MODE_CKZG_LE, 2 = MODE_DENEB (launch_batch_challenge)
inline int bch_wire_flags(int wire) { return wire == 1 ? BCH_LE : wire == 2 ? BCH_BE_HDR : 0; }

// One SHA-256 stream over the 64-byte blocks [blk0, blk1) of the message: the warp expands message schedules in
// parallel, lane 0 runs the rounds.  State carried in `state` between calls (BCH_INIT: start from the SHA-256 IV;
// BCH_FINAL: also absorb everything after blk1 -- the remaining full blocks and the padded tail -- and write r to
// r_out from lane 0).  tuples must be 32-byte aligned.  wk (64 x 32 words) and head (32 bytes) are shared memory.
__device__ __forceinline__ void batch_challenge_warp(uint32_t* __restrict__ r_out, Sha256State* __restrict__ state, const uint8_t* __restrict__ tuples,
                                                     unsigned long long n_total, int blk0, int blk1, int flags, uint32_t* wk, uint8_t* head) {
  const int lane = threadIdx.x;
  if (lane == 0) {
    const char dom[17] = "RCKZGBATCH___V1_";
    for (int i = 0; i < 16; i++) head[i] = (uint8_t)dom[i];
    for (int i = 0; i < 8; i++) head[16 + i] = 0;
    if (flags & BCH_BE_HDR) {   // MODE_DENEB: be64(4096) || be64(n)
      head[22] = 0x10;
      for (int i = 0; i < 8; i++) head[24 + i] = (uint8_t)(n_total >> (8 * (7 - i)));
    } else {
      head[17] = 0x10;  // le64(4096)
      for (int i = 0; i < 8; i++) head[24 + i] = (uint8_t)(n_total >> (8 * i));
    }
  }
  __syncwarp();
  const unsigned long long total = 32ull + 160ull * n_total;
  const int nfull = (int)(total / 64);
  if (flags & BCH_FINAL) blk1 = nfull;
  auto byte_at = [&](unsigned long long off) -> uint8_t { return off < 32 ? head[off] : tuples[off - 32]; };
  Sha256State s;
  if (flags & BCH_INIT) sha256_init(s); else s = *state;
  sha256_warp_blocks(s, blk1 - blk0, [&](int rel, uint32_t* w) {
    const int blk = blk0 + rel;
    unsigned long long off = 64ull * blk;
    if (blk >= 1) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(tuples + (off - 32));  // 32-byte aligned
      for (int i = 0; i < 16; i++) w[i] = bswap32(src[i]);
    } else {
      for (int i = 0; i < 16; i++)
        w[i] = ((uint32_t)byte_at(off + 4 * i) << 24) | ((uint32_t)byte_at(off + 4 * i + 1) << 16) | ((uint32_t)byte_at(off + 4 * i + 2) << 8) | byte_at(off + 4 * i + 3);
    }
  }, wk);
  if (lane != 0) return;
  if (!(flags & BCH_FINAL)) { *state = s; return; }
  uint32_t w[16];
  unsigned long long off = 64ull * nfull;
  uint8_t tail[128];
  int rem = (int)(total - off);
  for (int i = 0; i < rem; i++) tail[i] = byte_at(off + i);
  tail[rem] = 0x80;
  int tl = (rem + 9 <= 64) ? 64 : 128;
  for (int i = rem + 1; i < tl; i++) tail[i] = 0;
  unsigned long long bits = total * 8ull;
  for (int i = 0; i < 8; i++) tail[tl - 1 - i] = (uint8_t)(bits >> (8 * i));
  for (int o = 0; o < tl; o += 64) {
    for (int i = 0; i < 16; i++)
      w[i] = ((uint32_t)tail[o + 4 * i] << 24) | ((uint32_t)tail[o + 4 * i + 1] << 16) | ((uint32_t)tail[o + 4 * i + 2] << 8) | tail[o + 4 * i + 3];
    sha256_compress(s, w);
  }
  const int le = flags & BCH_LE;
  Fr r;
  for (int i = 0; i < 8; i++) r.l[i] = le ? bswap32(s.h[i]) : s.h[7 - i];
  mod_reduce_small<FrCfg, 2>(r.l);
  for (int i = 0; i < 8; i++) r_out[i] = r.l[i];
}

}  // namespace lw
