// Bucket MSM over Bandersnatch (twisted Edwards, extended coordinates) whose result is only tested for the identity: the
// random linear combination of a batch of Pedersen proofs (vrfs_pedersen_batch_verify, DESIGN §4 "Pedersen batch verification").
//
// Pipeline (all on the context's stream; the sort is the curve-independent one of csrc/msm.cuh):
//   k_msm_histogram / k_msm_scan / k_msm_scatter   signed radix-2^c digits, stateless plan (one column, segment = window)
//   k_te_msm_accumulate    tpb threads per bucket: te_madd of affine-cached records (complete on the prime-order subgroup, so
//                          there are no exceptional cases), then a shared-memory tree of te_add over the tpb partial sums
//   k_te_msm_chunks        one thread per run of TE_MSM_CHUNK buckets of a window: sum_j j*B_j of the run by a running sum,
//                          plus (run offset) * (sum of the run)
//   k_te_msm_window_sum    one block per window: the sum of its runs
//   k_te_msm_final         one thread: Horner over the windows, identity test, AND with the "bad input" flag -> verdict byte
//
// No oversized-bucket path: every scalar of the combination is a product with a secret uniform coefficient (or the coefficient
// itself), so the digits are uniform and the plan's window size leaves no window with only a few live buckets (te_msm_plan).
// A bucket above the plan's expected load is still summed correctly, only more slowly.
#pragma once
#include "msm.cuh"

namespace vrfs {

typedef TEPoint<BandCurve> BandPt;
typedef TEAffCached<BandCurve> BandAff;     // (x, y, d*x*y), Montgomery form: what te_madd reads

#ifndef VRFS_PED_BATCH_C
// 253-bit scalars (below r) and 127-bit coefficients: 253 mod 16 = 13 and 127 mod 16 = 15, so the top window of either kind of
// scalar keeps 2^12 - 2^14 live buckets.  c = 13, 14, 15 or 17 leave one of the two with 1-8 bits (2^0 - 2^7 buckets collecting a
// whole column's entries), which is why the window size does not follow the batch size.
#define VRFS_PED_BATCH_C 16
#endif
#define TE_MSM_CHUNK 16                     // buckets per thread of k_te_msm_chunks
#define TE_MSM_WSUM_THREADS 256

VRFS_HD inline MsmPlan te_msm_plan(uint32_t n) {
  MsmPlan p = msm_plan(n, 1, 0, VRFS_PED_BATCH_C, 0, 253);
  p.big = 0xffffffffu;                      // k_msm_scan lists no bucket as oversized
  return p;
}

HD_INLINE void band_aff_from_xy(BandAff& a, const BandCurve::F& x, const BandCurve::F& y) { a.x = x; a.y = y; a.dt = x * y * BandCurve::d(); }

__global__ void __launch_bounds__(128, MSM_ACC_MINBLOCKS) k_te_msm_accumulate(MsmPlan p, const BandAff* bases, const uint32_t* counts, const uint32_t* offsets,
                                                                             const uint32_t* list, BandPt* buckets) {
  __shared__ uint4 sh_raw[128 * sizeof(BandPt) / 16];
  BandPt* sh = reinterpret_cast<BandPt*>(sh_raw);
  const size_t nbuckets = (size_t)p.windows * p.nb;
  const uint32_t lane = threadIdx.x % p.tpb;
  const size_t b = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / p.tpb;
  const bool live = b < nbuckets;
  const uint32_t cnt = live ? counts[b] : 0u;
  BandPt acc; te_set_identity(acc);
  if (cnt) {
    const uint32_t* l = list + (b / p.nb) * (size_t)p.n + offsets[b];
    for (uint32_t j = lane; j < cnt; j += (uint32_t)p.tpb) {
      const uint32_t e = l[j];
      BandAff q; copy_words16(&q, bases + (e & 0x7fffffffu));
      if (j + p.tpb < cnt) prefetch_l1(bases + (l[j + p.tpb] & 0x7fffffffu), (unsigned)sizeof(BandAff));
      te_madd<BandCurve>(&acc, &acc, &q, (e >> 31) != 0, true);
    }
  }
  if (p.tpb > 1) {                          // block-uniform: the tpb partial sums of every bucket of the block, pairwise
    copy_words16(&sh[threadIdx.x], &acc);
    __syncthreads();
    for (int stride = p.tpb >> 1; stride > 0; stride >>= 1) {
      if ((int)lane < stride) { BandPt y; copy_words16(&y, &sh[threadIdx.x + stride]); te_add<BandCurve>(&acc, &acc, &y); copy_words16(&sh[threadIdx.x], &acc); }
      __syncthreads();
    }
  }
  if (live && lane == 0) copy_words16(&buckets[b], &acc);
}

// out[w * runs + k] = sum_{j < CHUNK} (k CHUNK + j + 1) B[w][k CHUNK + j]   (bucket index j holds the digit magnitude j + 1)
__global__ void __launch_bounds__(128) k_te_msm_chunks(MsmPlan p, const BandPt* buckets, BandPt* out) {
  const uint32_t runs = (uint32_t)p.nb / TE_MSM_CHUNK;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (uint32_t)p.windows * runs) return;
  const uint32_t w = t / runs, k = t % runs;
  const BandPt* B = buckets + (size_t)w * p.nb + (size_t)k * TE_MSM_CHUNK;
  BandPt S, T, y;
  te_set_identity(S); te_set_identity(T);
  for (int j = TE_MSM_CHUNK - 1; j >= 0; j--) {        // S = B[j] + ... + B[CHUNK-1];  T += S  ->  T = sum (j + 1) B[j]
    copy_words16(&y, &B[j]);
    te_add<BandCurve>(&S, &S, &y);
    te_add<BandCurve>(&T, &T, &S);
  }
  const uint32_t m = k * TE_MSM_CHUNK;                  // + m S, double-and-add over the bits of the public run offset
  BandPt Q; te_set_identity(Q);
  for (int bit = 31 - __clz((int)(m | 1u)); bit >= 0; bit--) {
    te_dbl<BandCurve>(&Q, &Q, true);
    if ((m >> bit) & 1u) te_add<BandCurve>(&Q, &Q, &S);
  }
  te_add<BandCurve>(&T, &T, &Q);
  copy_words16(&out[t], &T);
}

// one block per window: wsum[w] = sum of the window's runs
__global__ void __launch_bounds__(TE_MSM_WSUM_THREADS) k_te_msm_window_sum(MsmPlan p, const BandPt* runs_in, BandPt* wsum) {
  __shared__ uint4 sh_raw[TE_MSM_WSUM_THREADS * sizeof(BandPt) / 16];
  BandPt* sh = reinterpret_cast<BandPt*>(sh_raw);
  const uint32_t runs = (uint32_t)p.nb / TE_MSM_CHUNK;
  const BandPt* R = runs_in + (size_t)blockIdx.x * runs;
  BandPt acc, y; te_set_identity(acc);
  for (uint32_t k = threadIdx.x; k < runs; k += TE_MSM_WSUM_THREADS) { copy_words16(&y, &R[k]); te_add<BandCurve>(&acc, &acc, &y); }
  copy_words16(&sh[threadIdx.x], &acc);
  __syncthreads();
  for (int s = TE_MSM_WSUM_THREADS / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) { copy_words16(&y, &sh[threadIdx.x + s]); te_add<BandCurve>(&acc, &acc, &y); copy_words16(&sh[threadIdx.x], &acc); }
    __syncthreads();
  }
  if (threadIdx.x == 0) copy_words16(&wsum[blockIdx.x], &acc);
}

// verdict = (sum_w 2^(c w) wsum[w] is the identity) && !*bad.  X = 0 and Y = Z is exact on the odd-order subgroup (the 2-torsion
// point (0, -1) also has X = 0 but Y = -Z); points outside the subgroup have already set *bad.
__global__ void __launch_bounds__(32) k_te_msm_final(MsmPlan p, const BandPt* wsum, const uint32_t* bad, uint8_t* verdict) {
  if (threadIdx.x != 0) return;
  BandPt acc, y;
  copy_words16(&acc, &wsum[p.windows - 1]);
  for (int w = p.windows - 2; w >= 0; w--) {
    for (int k = 0; k < p.c; k++) te_dbl<BandCurve>(&acc, &acc, true);
    copy_words16(&y, &wsum[w]);
    te_add<BandCurve>(&acc, &acc, &y);
  }
  *verdict = (uint8_t)(te_is_identity(acc) && *bad == 0u);
}

}  // namespace vrfs
