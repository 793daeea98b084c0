// TEST INFRASTRUCTURE ONLY: the KZG opening quotient (csrc/kzg_open.cuh) compiled for the HOST and run through the three phases of
// the kernels of csrc/kzg.cuh for one polynomial - segment values and the block suffix scan (warp shuffles emulated lane by lane),
// the chunk carries, and the finish.  Built by tests/test_host_emul_kzg.py into a temporary directory; nothing in the product
// links this file.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../../ark_ec_vrfs_b200/csrc/gen/field_consts.cuh"
#include "../../ark_ec_vrfs_b200/csrc/kzg_open.cuh"
using namespace vrfs;

static Fr255 load_mont(const uint8_t* p) {           // what the kernels' fr_load_reduced + to_mont do
  uint32_t raw[8];
  load_le<8>(raw, p);
  cond_sub_p<BlsFr>(raw, 0u); cond_sub_p<BlsFr>(raw, 0u);
  return to_mont<BlsFr>(raw);
}
static void store_canonical(uint8_t* p, const Fr255& a) { uint32_t raw[8]; from_mont<BlsFr>(raw, a); store_le<8>(p, raw); }

extern "C" int hostemu_kzg_chunk() { return KZG_OPEN_CH; }

// p = sum_{j < len} coeffs[32 j ..] X^j at z: out_v = p(z), out_q = the n >= len rows of the quotient's MSM column (zeros from
// len - 1 on), both canonical 32-byte LE
extern "C" void hostemu_kzg_open(uint32_t len, uint32_t n, const uint8_t* coeffs, const uint8_t* zb, uint8_t* out_v, uint8_t* out_q) {
  const uint32_t chunks = len ? (len + KZG_OPEN_CH - 1) / KZG_OPEN_CH : 1;
  const Fr255 z = load_mont(zb);
  auto coeff = [&](uint32_t j) { return j < len ? load_mont(coeffs + (size_t)32 * j) : Fr255::zero(); };
  std::vector<Fr255> agg(chunks), carry(chunks);
  std::vector<KzgSpan> seg((size_t)chunks * KZG_OPEN_THREADS);
  // phase 1 (k_kzg_quotient_chunks)
  for (uint32_t c = 0; c < chunks; c++) {
    KzgSpan s[KZG_OPEN_THREADS];
    for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) {
      const uint32_t base = c * KZG_OPEN_CH + KZG_OPEN_SEG * t;
      s[t] = {kzg_segment_value(z, [&](int m) { return coeff(base + m); }), kzg_pow2k(z, KZG_OPEN_LOG_SEG)};
    }
    for (unsigned d = 1; d < 32; d <<= 1) {                    // every lane reads the value of lane + d before any lane writes
      KzgSpan up[KZG_OPEN_THREADS];
      for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) up[t] = (t & 31u) + d < 32 ? s[t + d] : s[t];
      for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) if ((t & 31u) + d < 32) s[t] = kzg_span_combine(s[t], up[t]);
    }
    for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) {
      const uint32_t w = t >> 5;
      KzgSpan ex = (t & 31u) == 31 ? kzg_span_identity() : s[t + 1];
      KzgSpan above = kzg_span_identity();
      for (int u = KZG_OPEN_THREADS / 32 - 1; u > (int)w; u--) above = kzg_span_combine(s[32 * u], above);
      seg[(size_t)c * KZG_OPEN_THREADS + t] = kzg_span_combine(ex, above);
      if (t == 0) agg[c] = kzg_span_combine(s[0], above).h;
    }
  }
  // phase 2 (k_kzg_quotient_carry)
  const KzgSpan step = {Fr255::zero(), kzg_pow2k(z, KZG_OPEN_LOG_CH)};
  Fr255 k = Fr255::zero();
  carry[chunks - 1] = k;
  for (uint32_t c = chunks - 1; c-- > 0;) { KzgSpan e = step; e.h = agg[c + 1]; carry[c] = k = kzg_carry_in(e, k); }
  // phase 3 (k_kzg_quotient_finish)
  const uint32_t grid = (n + KZG_OPEN_CH - 1) / KZG_OPEN_CH;
  for (uint32_t c = 0; c < grid; c++)
    for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) {
      const uint32_t base = c * KZG_OPEN_CH + KZG_OPEN_SEG * t;
      auto store = [&](int m, const Fr255& q) { if (base + m < n) store_canonical(out_q + (size_t)32 * (base + m), q); };
      if (c >= chunks) { for (int m = 0; m < KZG_OPEN_SEG; m++) store(m, Fr255::zero()); continue; }
      const Fr255 in = kzg_carry_in(seg[(size_t)c * KZG_OPEN_THREADS + t], carry[c]);
      const Fr255 v = kzg_segment_finish(z, in, [&](int m) { return coeff(base + m); }, store);
      if (base == 0) store_canonical(out_v, v);
    }
}
