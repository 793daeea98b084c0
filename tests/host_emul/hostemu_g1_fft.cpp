// TEST INFRASTRUCTURE ONLY: the G1 FFT (csrc/g1_fft.cuh) compiled for the HOST - the twiddle multiplication, the whole transform
// played stage by stage with the kernels' index arithmetic (load at the bit-reversed index, one butterfly per thread per stage,
// the [1/n] scaling and the per-block batch-affine store), and the batch-affine store alone.  Built by tests/test_host_emul_g1_fft.py
// into a temporary directory; nothing in the product links this file.
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <vector>
#include "../../ark_ec_vrfs_b200/csrc/gen/field_consts.cuh"
#include "../../ark_ec_vrfs_b200/csrc/g1_fft.cuh"
using namespace vrfs;

// what k_g1_fft_store does for the points [base, base + count) of one block
static void store_block(uint8_t* out, G1Pt* pts, uint32_t count) {
  Fq381 z[G1_FFT_STORE_THREADS], pre[G1_FFT_STORE_THREADS];
  for (uint32_t t = 0; t < count; t++) z[t] = pts[t].Z;
  g1_fft_batch_inv(z, pre, count);
  for (uint32_t t = 0; t < count; t++) g1_fft_store_one(out + (size_t)96 * t, pts[t], z[t]);
}
static void store_all(uint8_t* out, std::vector<G1Pt>& pts) {
  for (size_t base = 0; base < pts.size(); base += G1_FFT_STORE_THREADS) {
    const uint32_t count = (uint32_t)std::min<size_t>(pts.size() - base, G1_FFT_STORE_THREADS);
    store_block(out + 96 * base, &pts[base], count);
  }
}

extern "C" int hostemu_g1_fft_store_threads() { return G1_FFT_STORE_THREADS; }

// out = [w] P: P 96-byte affine LE in G1, w canonical 32-byte LE < r
extern "C" void hostemu_g1_mul(const uint8_t* p, const uint8_t* w, uint8_t* out) {
  uint32_t k[8];
  load_le<8>(k, w);
  std::vector<G1Pt> r(1);
  G1Pt P;
  g1_fft_load_one(P, p);
  g1_fft_mul(&r[0], &P, k);
  store_all(out, r);
}

// vrfs_g1_fft_batch on the host: 2^logn points in, 2^logn points out (96-byte affine LE)
extern "C" void hostemu_g1_fft(int logn, int inverse, const uint8_t* in, uint8_t* out) {
  const uint32_t n = 1u << logn, half_n = n / 2;
  std::vector<Fr255> tw(half_n + 1);                              // k_ntt_twiddles
  for (uint32_t j = 0; j < half_n; j++) tw[j] = fr_pow_u32(ntt_domain_gen(logn, inverse != 0), j);
  tw[half_n] = fr_pow_u32(ntt_const(2), (uint32_t)logn);
  std::vector<G1Pt> work(n);
  for (uint32_t i = 0; i < n; i++) {                              // k_g1_fft_load
    uint32_t rev = 0;
    for (int b = 0; b < logn; b++) rev |= ((i >> b) & 1u) << (logn - 1 - b);
    g1_fft_load_one(work[rev], in + (size_t)96 * i);
  }
  for (int s = 1; s <= logn; s++)                                 // k_g1_fft_stage
    for (uint32_t u = 0; u < half_n; u++) {
      const uint32_t half = 1u << (s - 1), k = (u >> (s - 1)) << s, j = u & (half - 1);
      g1_fft_butterfly(&work[k + j], &work[k + j + half], tw[(size_t)j * (half_n >> (s - 1))], j == 0);
    }
  if (inverse)                                                    // k_g1_fft_store
    for (uint32_t i = 0; i < n; i++) g1_fft_mul_mont(&work[i], &work[i], tw[half_n]);
  store_all(out, work);
}

// the batch-affine store alone: n projective points, X | Y | Z canonical 48-byte LE each (identity: Z = 0) -> affine LE
extern "C" void hostemu_g1_batch_affine(uint32_t n, const uint8_t* proj, uint8_t* out) {
  std::vector<G1Pt> pts(n);
  for (uint32_t i = 0; i < n; i++) {
    uint32_t raw[12];
    load_le<12>(raw, proj + (size_t)144 * i); pts[i].X = to_mont<BlsFq>(raw);
    load_le<12>(raw, proj + (size_t)144 * i + 48); pts[i].Y = to_mont<BlsFq>(raw);
    load_le<12>(raw, proj + (size_t)144 * i + 96); pts[i].Z = to_mont<BlsFq>(raw);
  }
  store_all(out, pts);
}
