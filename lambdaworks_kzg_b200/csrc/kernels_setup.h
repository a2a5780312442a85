#pragma once
#include "kernels.h"
namespace lw {
void launch_setup_decode_g1(void* d_canon24, int* d_status, const void* d_in48, int n, cudaStream_t st);
void launch_setup_decode_g2(void* d_canon48, int* d_status, const void* d_in96, int n, cudaStream_t st);
// c-kzg-4844 setups: strict G2 decoding (canonical x, no infinity, on the twist, in G2); status 0 ok, 1 encoding,
// 2 not on the twist, 3 not in G2
void launch_setup_decode_g2_strict(void* d_canon48, int* d_status, const void* d_in96, int n, cudaStream_t st);
// rho = SHA-256 of nblocks already padded 64-byte blocks, read big-endian, mod r (8 u32 canonical).  One warp.
void launch_setup_rho(void* d_rho, const void* d_msg, int nblocks, cudaStream_t st);
// d_sc[k] = rho^k (8 u32 canonical, k < 4096); d_blob = the MODE_DENEB blob (4096 x 32 bytes) with value rho^k at w^k
void launch_setup_rho_powers(void* d_sc, void* d_blob, const void* d_rho, cudaStream_t st);
// d_sc[j] = -d_coef[j] (4096 Montgomery Fr in, canonical out)
void launch_setup_neg_coef(void* d_sc, const void* d_coef, cudaStream_t st);
}  // namespace lw
