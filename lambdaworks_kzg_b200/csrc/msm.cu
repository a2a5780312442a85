// Batched fixed-base G1 MSM over the 4096-point SRS: the commitment / proof
// hot loop (replaces lambdaworks-math `msm::pippenger::msm` as called by
// KZG::commit / KZG::open -- /root/reference/src/lib.rs:241-243, 269-270, 329,
// 394; SURVEY §3.1/§3.2).
//
// B200-first design: the SRS never changes, and the GPU has 180 GB of HBM, so
// instead of per-call bucket accumulation + bucket reduction we precompute the
// FULL signed-digit table of the 128-bit GLV halves (csrc/recode.cuh)
//        T[j][i][d-1] = d * 2^(c j) * P_i ,  j < W = ceil(128 / c)          (affine, 96 B)
// once at setup (c = 16: 8 windows, 100 GiB) and an MSM becomes
//        C = sum_{i,j} sign(d_ij) T[j][i][|d_ij|-1]  +  psi( sum_{i,j} sign(e_ij) T[j][i][|e_ij|-1] )
// with k_i = m_i + q_i x^2, d = digits of m_i, e = digits of q_i, psi(X, Y) = (beta X, -Y) = [x^2](X, Y):
// 4096 * 2 W additions with NO buckets, NO sorting, NO reduction tree over buckets and perfectly uniform work per
// thread.  The lower half of every block's threads sums the m-halves, the upper half the q-halves; psi is applied
// once, where the two meet in the block reduction.  Each thread owns a slice of points, streams their scalars with
// 128-bit loads, splits and recodes them in registers, gathers the table entries (3 x 32 B sectors each, random
// in HBM/L2) and accumulates; a block-level tree in shared memory and a tiny finalize kernel combine the
// per-thread sums.  The kernels are bound by the integer (IMAD) pipe.
#include "msm_common.cuh"

namespace lw {

int msm_threads_per_block() { return MSM_THREADS; }

template <bool BE>
__global__ void __launch_bounds__(MSM_THREADS, LWKZG_MSM_MIN_BLOCKS)
msm_gather_kernel(G1Xyzz* __restrict__ partials, const uint4* __restrict__ table, const uint8_t* __restrict__ scalars,
                  int c, int nwin, uint32_t cnt_top, int pt_threads, int wsplit) {
  constexpr int HT = MSM_THREADS / 2;
  __shared__ uint32_t sk[4][MSM_THREADS];
  __shared__ uint32_t red[48 * HT];

  const int tid = threadIdx.x;
  const int half = tid / HT;
  const int blob = blockIdx.y;
  const int q = blockIdx.x * HT + (tid % HT);
  const int pl = q % pt_threads;   // point lane
  const int wg = q / pt_threads;   // window group (only > 0 for tiny batches)
  const uint8_t* sc = scalars + (size_t)blob * BLOB_BYTES;
  auto limb = [&](int w) { return sk[w][tid]; };

  G1Xyzz acc = xyzz_inf();

  for (int pi = pl; pi < N_POINTS; pi += pt_threads) {
    uint32_t h4[4];
    load_scalar_half<BE>(h4, sc, pi, half);
#pragma unroll
    for (int i = 0; i < 4; i++) sk[i][tid] = h4[i];   // private column: no sync needed
    // ---- recode on the fly, gather, accumulate; the entry for window j+1 is
    // requested before the mixed addition for window j is issued.
    int carry = 0;
    int d = 0;
    G1Affine cur = g1a_inf();
    for (int j = 0; j <= nwin; j++) {
      int dn = 0;
      G1Affine nxt = g1a_inf();
      if (j < nwin) {
        dn = glv_digit(limb, c, nwin, j, carry);
        if ((j % wsplit) != wg) dn = 0;
        if (dn != 0) nxt = load_entry(table, entry_index(c, nwin, cnt_top, j, pi, dn < 0 ? -dn : dn));
      }
      if (d != 0) {
        cur.y = fp_cneg(cur.y, d < 0);
        xyzz_madd_hot(acc, cur);
      }
      cur = nxt; d = dn;
    }
  }

  block_reduce_xyzz_glv<MSM_THREADS>(acc, red);
  if (tid == 0) partials[(size_t)blob * gridDim.x + blockIdx.x] = acc;
}

// variant = accumulators per thread (K), threads per blob (= block size) and register budget
void launch_msm_gather(void* d_partials, const void* d_table, int c, const void* d_scalars, bool be_input, int n_blobs,
                       int blocks_per_blob, cudaStream_t st);
// defined in msm_ba_v*.cu (one translation unit per variant)
#define LW_BA_DECL(N) void launch_ba_v##N(void*, const void*, int, const void*, bool, int, void*, cudaStream_t, int)
LW_BA_DECL(0); LW_BA_DECL(1);
struct BaVariant { int k, threads; };
static const BaVariant BA_VARIANTS[] = {{64, 128}, {64, 64}};   // keep in step with msm_ba_v*.cu
constexpr int N_BA_VARIANTS = (int)(sizeof(BA_VARIANTS) / sizeof(BA_VARIANTS[0]));
static int g_ba_variant = 0;
void msm_ba_set_variant(int v) { if (v >= 0 && v < N_BA_VARIANTS) g_ba_variant = v; }
int msm_ba_num_variants() { return N_BA_VARIANTS; }
int msm_ba_variant() { return g_ba_variant; }
int msm_ba_threads() { return BA_VARIANTS[g_ba_variant].threads; }
int msm_ba_slots() { return BA_VARIANTS[g_ba_variant].k; }
size_t msm_ba_scratch_bytes(int n_blobs) {   // sized for the largest variant: 64 slots x 9 words x 128 threads
  return (size_t)n_blobs * 64 * 9 * 128 * sizeof(uint4);
}

// one block per blob (blobs on grid.x: no 65535 limit); partials: one XYZZ per blob
void launch_msm_gather_ba(void* d_partials, const void* d_table, int c, const void* d_scalars, bool be_input, int n_blobs,
                          void* d_scratch, cudaStream_t st, int split) {
  if (n_blobs <= 0) return;
  if (glv_num_windows(c) > BA_VARIANTS[g_ba_variant].k) {   // tiny windows: a round could not hold one point's digits
    launch_msm_gather(d_partials, d_table, c, d_scalars, be_input, n_blobs, split, st);
    return;
  }
  switch (g_ba_variant) {
    case 1: launch_ba_v1(d_partials, d_table, c, d_scalars, be_input, n_blobs, d_scratch, st, split); break;
    default: launch_ba_v0(d_partials, d_table, c, d_scalars, be_input, n_blobs, d_scratch, st, split); break;
  }
  count_launch();
}

// Sum the per-block partials of one blob, normalise (one inversion), compress.
__global__ void __launch_bounds__(32)
msm_finalize_kernel(uint8_t* __restrict__ out48, G1Affine* __restrict__ aff_out, const G1Xyzz* __restrict__ partials,
                    int parts, int n) {
  const int blob = blockIdx.x * blockDim.x + threadIdx.x;
  if (blob >= n) return;
  const G1Xyzz* p = partials + (size_t)blob * parts;
  G1Xyzz acc = p[0];
  for (int i = 1; i < parts; i++) {
    G1Xyzz o = p[i];
    xyzz_add_ni(acc, o);
  }
  G1Affine a = xyzz_to_affine(acc);
  if (aff_out) aff_out[blob] = a;
  if (out48) g1_compress(out48 + (size_t)blob * 48, a);
}

void launch_msm_gather(void* d_partials, const void* d_table, int c, const void* d_scalars, bool be_input, int n_blobs,
                       int blocks_per_blob, cudaStream_t st) {
  if (n_blobs <= 0) return;
  // each block carries MSM_THREADS / 2 point lanes per GLV half; once every point has its own lane the windows
  // are split across the remaining lanes
  const int total = blocks_per_blob * (MSM_THREADS / 2);
  const int pt = total < N_POINTS ? total : N_POINTS;
  const int ws = total / pt;
  const int nwin = glv_num_windows(c);
  const uint32_t cnt_top = glv_top_max(c) + 1u;
  for (int b0 = 0; b0 < n_blobs; b0 += 65535) {   // gridDim.y limit
    const int nb = n_blobs - b0 < 65535 ? n_blobs - b0 : 65535;
    dim3 grid(blocks_per_blob, nb);
    G1Xyzz* part = (G1Xyzz*)d_partials + (size_t)b0 * blocks_per_blob;
    const uint8_t* sc = (const uint8_t*)d_scalars + (size_t)b0 * BLOB_BYTES;
    if (be_input)
      msm_gather_kernel<true><<<grid, MSM_THREADS, 0, st>>>(part, (const uint4*)d_table, sc, c, nwin, cnt_top, pt, ws);
    else
      msm_gather_kernel<false><<<grid, MSM_THREADS, 0, st>>>(part, (const uint4*)d_table, sc, c, nwin, cnt_top, pt, ws);
  }
  count_launch();
}

// Warp-per-blob variant for many partials (single-blob / tiny-batch calls use up to
// 128 blocks per blob): lanes sum strided partials, then a 5-level tree in shared memory.
__global__ void __launch_bounds__(32) msm_finalize_warp_kernel(uint8_t* __restrict__ out48, G1Affine* __restrict__ aff_out,
                                                                const G1Xyzz* __restrict__ partials, int parts, int n) {
  __shared__ uint32_t red[48 * 16];
  const int blob = blockIdx.x, lane = threadIdx.x;
  const G1Xyzz* p = partials + (size_t)blob * parts;
  G1Xyzz acc = xyzz_inf();
  for (int i = lane; i < parts; i += 32) {
    G1Xyzz o = p[i];
    xyzz_add_ni(acc, o);
  }
  for (int s = 16; s > 0; s >>= 1) {
    if (lane >= s && lane < 2 * s) xyzz_to_smem(red, 16, lane - s, acc);
    __syncwarp();
    if (lane < s) {
      G1Xyzz o = xyzz_from_smem(red, 16, lane);
      xyzz_add_ni(acc, o);
    }
    __syncwarp();
  }
  if (lane == 0) {
    G1Affine a = xyzz_to_affine(acc);
    if (aff_out) aff_out[blob] = a;
    if (out48) g1_compress(out48 + (size_t)blob * 48, a);
  }
}

void launch_msm_finalize(void* d_out48, void* d_aff_out, const void* d_partials, int parts_per_blob, int n_blobs, cudaStream_t st) {
  if (n_blobs <= 0) return;
  if (parts_per_blob >= 8)
    msm_finalize_warp_kernel<<<n_blobs, 32, 0, st>>>((uint8_t*)d_out48, (G1Affine*)d_aff_out, (const G1Xyzz*)d_partials, parts_per_blob, n_blobs);
  else
    msm_finalize_kernel<<<(n_blobs + 31) / 32, 32, 0, st>>>((uint8_t*)d_out48, (G1Affine*)d_aff_out, (const G1Xyzz*)d_partials, parts_per_blob, n_blobs);
  count_launch();
}

}  // namespace lw
