// The radix-2 FFT over BLS12-381 G1 (vrfs_g1_fft_batch): the transform of vrfs_fr_fft_batch with points in place of field
// elements, out_i = sum_j [w^(ij)] P_j (forward) or [1/n] sum_j [w^(-ij)] P_j (inverse), both sides in natural order.  The inverse
// transform of the monomial powers [tau^j] G1 is the Lagrange basis [L_i(tau)] G1 of the same domain (ring-proof's
// `RingBuilderKey::from_srs`, an arkworks `Radix2EvaluationDomain::ifft` over G1 projective points).
//   k_g1_fft_load   affine LE -> Montgomery projective at the bit-reversed index (identity -> (0 : 1 : 0))
//   k_ntt_twiddles  w^j, j < n/2, and 1/n (csrc/ring.cuh)
//   k_g1_fft_stage  one launch per stage of the decimation-in-time network, one thread per butterfly (a, b) <- (a + [w] b, a - [w] b)
//   k_g1_fft_store  [1/n] of every point (inverse), then projective -> canonical affine LE with one Fq inversion per block
// The twiddle multiplication [w] b splits w = k1 + q z^2 (g1_glv_split, both halves < 2^128) and computes k1 b + q (-phi(b)) with
// -phi(X : Y : Z) = (beta X : -Y : Z): one chain of 128 doublings shared by the two halves, signed digits of G1_FFT_WIN bits over one
// table of [d] b.  Every formula is complete: identities, equal points and a - t = 0 occur (the all-identity vector, tiled inputs).
// The per-thread pieces are host-compilable; tests/host_emul/hostemu_g1_fft.cpp runs the whole transform with them on the CPU.
#pragma once
#include "ring.cuh"

namespace vrfs {

#define G1_FFT_WIN 4                                              // signed window bits of the GLV halves (DESIGN.md, G1 FFT)
#define G1_FFT_TAB ((1 << (G1_FFT_WIN - 1)) + 1)                  // [d] b for d = 0 .. 2^(WIN-1)
#define G1_FFT_WINDOWS ((128 + G1_FFT_WIN) / G1_FFT_WIN)          // 128-bit halves + the top bit's carry window
#define G1_FFT_STAGE_THREADS 64
#define G1_FFT_STORE_THREADS 128                                  // points per Fq inversion in k_g1_fft_store

// signed digit of window w of a 128-bit scalar (4 limbs), in [-2^(WIN-1), 2^(WIN-1)]: bits [w WIN - 1, (w + 1) WIN) as
// d = b_(w WIN - 1) + sum_(i < WIN-1) b_(w WIN + i) 2^i - b_(w WIN + WIN - 1) 2^(WIN-1), so sum_w d_w 2^(w WIN) = k and every digit
// depends on its own bits only (no carry from the windows below: the doubling chain reads them top down)
HD_INLINE int g1_fft_digit(const uint32_t* k, int w) {
  const int pos = w * G1_FFT_WIN - 1;
  const uint32_t mask = (2u << G1_FFT_WIN) - 1u;
  uint32_t v;
  if (pos < 0) {
    v = (k[0] << 1) & mask;
  } else {
    const int limb = pos >> 5, sh = pos & 31;
    uint64_t x = limb < 4 ? k[limb] : 0u;
    if (limb + 1 < 4) x |= (uint64_t)k[limb + 1] << 32;
    v = (uint32_t)(x >> sh) & mask;
  }
  return (int)((v + 1u) >> 1) - (int)((v >> G1_FFT_WIN) << G1_FFT_WIN);
}
HD_INLINE Fq381 g1_fft_beta() { Fq381 b; for (int i = 0; i < 12; i++) b.v[i] = G1WireConsts::beta(i); return b; }

// r = [w] p for a canonical scalar w < r (8 limbs) and p in G1 (the GLV split is the endomorphism of G1); r may alias p
HD_INLINE void g1_fft_mul(G1Pt* r, const G1Pt* p, const uint32_t* w) {
  uint32_t k1[4], q[4];
  g1_glv_split(k1, q, w);
  G1Pt tab[G1_FFT_TAB];
  sw_set_identity(tab[0]);
  tab[1] = *p;
  g1_dbl(&tab[2], p);
  for (int d = 3; d < G1_FFT_TAB; d++) sw_add<G1Curve>(&tab[d], &tab[d - 1], p);
  const Fq381 beta = g1_fft_beta();
  G1Pt acc;
  sw_set_identity(acc);
#pragma unroll 1
  for (int win = G1_FFT_WINDOWS - 1; win >= 0; win--) {
    if (win != G1_FFT_WINDOWS - 1)
      for (int i = 0; i < G1_FFT_WIN; i++) g1_dbl(&acc, &acc);
    const int d1 = g1_fft_digit(k1, win), d2 = g1_fft_digit(q, win);
    G1Pt t = tab[d1 < 0 ? -d1 : d1];
    sw_cneg(t, d1 < 0);
    sw_add<G1Curve>(&acc, &acc, &t);
    t = tab[d2 < 0 ? -d2 : d2];                                    // [d2] (-phi(p)) = (beta X : -Y : Z) of [d2] p
    t.X = t.X * beta;
    sw_cneg(t, d2 >= 0);
    sw_add<G1Curve>(&acc, &acc, &t);
  }
  *r = acc;
}
HD_INLINE void g1_fft_mul_mont(G1Pt* r, const G1Pt* p, const Fr255& w) {   // the same with w in Montgomery form (a twiddle)
  uint32_t raw[8];
  from_mont<BlsFr>(raw, w);
  g1_fft_mul(r, p, raw);
}
// one butterfly of the decimation-in-time network, (a, b) <- (a + t, a - t) with t = [w] b; unit (w = 1, j = 0): t = b
HD_INLINE void g1_fft_butterfly(G1Pt* a, G1Pt* b, const Fr255& w, bool unit) {
  G1Pt t = *b, s;
  if (!unit) g1_fft_mul_mont(&t, b, w);
  sw_add<G1Curve>(&s, a, &t);
  sw_cneg(t, true);
  sw_add<G1Curve>(b, a, &t);
  *a = s;
}
// 96-byte affine LE (zeros = identity) -> Montgomery projective
HD_INLINE void g1_fft_load_one(G1Pt& P, const uint8_t* in) {
  uint32_t raw[12];
  G1Aff a;
  load_le<12>(raw, in); a.x = to_mont<BlsFq>(raw);
  load_le<12>(raw, in + 48); a.y = to_mont<BlsFq>(raw);
  g1_load_aff(P, &a, false);
}
// Montgomery's trick over the Z of one block: z[i] <- 1/z[i] for the count values, with one inversion; z = 0 (the identity) is left
// out of the chain and stays 0.  pre: count values of scratch (the prefix products)
HD_INLINE void g1_fft_batch_inv(Fq381* z, Fq381* pre, uint32_t count) {
  Fq381 acc = Fq381::one();
  for (uint32_t i = 0; i < count; i++) {
    pre[i] = acc;
    if (!z[i].is_zero()) acc = acc * z[i];
  }
  Fq381 inv = fq381_inv_fast(acc);                                 // 1 / (product of the non-zero z)
  for (uint32_t i = count; i-- > 0;) {
    if (z[i].is_zero()) continue;
    const Fq381 zi = inv * pre[i];
    inv = inv * z[i];
    z[i] = zi;
  }
}
// projective P with zi = 1/Z (0 for the identity) -> canonical affine LE; the identity is 96 zero bytes
HD_INLINE void g1_fft_store_one(uint8_t* out, const G1Pt& P, const Fq381& zi) {
  uint32_t raw[12];
  from_mont<BlsFq>(raw, P.X * zi); store_le<12>(out, raw);
  from_mont<BlsFq>(raw, P.Y * zi); store_le<12>(out + 48, raw);
}

#ifdef __CUDACC__
__global__ void k_g1_fft_load(int logn, const uint8_t* in, G1Pt* work) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, n = 1u << logn;
  if (i >= n) return;
  G1Pt P;
  g1_fft_load_one(P, in + (size_t)96 * i);
  const uint32_t rev = logn ? __brev(i) >> (32 - logn) : 0u;
  copy_words16(work + rev, &P);
}
// stage s (1-based) of the network on bit-reversed input, as k_ntt_stage: butterfly u pairs k + j and k + j + 2^(s-1)
__global__ void __launch_bounds__(G1_FFT_STAGE_THREADS) k_g1_fft_stage(int logn, int s, const Fr255* tw, G1Pt* work) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x, half_n = (1u << logn) / 2u;
  if (u >= half_n) return;
  const uint32_t half = 1u << (s - 1), k = (u >> (s - 1)) << s, j = u & (half - 1);
  G1Pt a, b;
  copy_words16(&a, work + k + j);
  copy_words16(&b, work + k + j + half);
  g1_fft_butterfly(&a, &b, tw[(size_t)j * (half_n >> (s - 1))], j == 0);
  copy_words16(work + k + j, &a);
  copy_words16(work + k + j + half, &b);
}
// the inverse transform's [1/n] (tw[n/2], k_ntt_twiddles), then canonical affine with one inversion per block of points
__global__ void __launch_bounds__(G1_FFT_STORE_THREADS) k_g1_fft_store(int logn, int inverse, const G1Pt* work, const Fr255* tw, uint8_t* out) {
  __shared__ Fq381 z[G1_FFT_STORE_THREADS], pre[G1_FFT_STORE_THREADS];
  const uint32_t n = 1u << logn, base = blockIdx.x * G1_FFT_STORE_THREADS, i = base + threadIdx.x;
  const uint32_t count = n - base < G1_FFT_STORE_THREADS ? n - base : G1_FFT_STORE_THREADS;
  G1Pt P;
  sw_set_identity(P);
  if (i < n) {
    copy_words16(&P, work + i);
    if (inverse) g1_fft_mul_mont(&P, &P, tw[n / 2]);
    z[threadIdx.x] = P.Z;
  }
  __syncthreads();
  if (threadIdx.x == 0) g1_fft_batch_inv(z, pre, count);
  __syncthreads();
  if (i < n) g1_fft_store_one(out + (size_t)96 * i, P, z[threadIdx.x]);
}
#endif  // __CUDACC__

}  // namespace vrfs
