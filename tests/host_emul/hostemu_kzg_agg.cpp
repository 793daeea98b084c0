// TEST INFRASTRUCTURE ONLY: the evaluation and aggregation of vrfs_kzg_open_aggregated_batch (csrc/kzg_open.cuh) compiled for the
// HOST and run the way the kernels of csrc/kzg.cuh run them - k_kzg_eval_chunks (segment values, the ordered warp reduction with
// its shuffles emulated lane by lane, then the warps in order), k_kzg_eval_finish (Horner over the chunks) and k_kzg_aggregate
// (one thread per segment of a group's rows).  Built by tests/test_host_emul_kzg_aggregated.py into a temporary directory;
// nothing in the product links this file.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../../ark_ec_vrfs_b200/csrc/gen/field_consts.cuh"
#include "../../ark_ec_vrfs_b200/csrc/kzg_open.cuh"
using namespace vrfs;

static Fr255 load_reduced(const uint8_t* p) {        // fr_load_reduced: the residue < r, not converted
  Fr255 a;
  load_le<8>(a.v, p);
  cond_sub_p<BlsFr>(a.v, 0u); cond_sub_p<BlsFr>(a.v, 0u);
  return a;
}
static Fr255 load_mont(const uint8_t* p) { return to_mont<BlsFr>(load_reduced(p).v); }
static void store_canonical(uint8_t* p, const Fr255& a) { uint32_t raw[8]; from_mont<BlsFr>(raw, a); store_le<8>(p, raw); }

extern "C" int hostemu_kzg_agg_chunk() { return KZG_OPEN_CH; }

// n_polys polynomials (coeff_off: n_polys + 1 coefficient offsets into coeffs) in n_groups groups (group_off), points zs, coefficients
// nus: out_values[i] = p_i(z_g(i)); out_rows = for each group, rows[g] .. of its longest polynomial's length (row_off: n_groups + 1),
// the aggregated coefficients sum nu_i a_ij; all canonical 32-byte LE
extern "C" void hostemu_kzg_agg(uint32_t n_groups, uint32_t n_polys, const uint64_t* group_off, const uint64_t* coeff_off, const uint8_t* coeffs,
                                const uint8_t* zs, const uint8_t* nus, uint8_t* out_values, const uint64_t* row_off, uint8_t* out_rows) {
  // the host tables of the entry point
  std::vector<uint32_t> chunk_off(n_polys + 1, 0), poly_group(n_polys), chunk_poly;
  for (uint32_t g = 0; g < n_groups; g++)
    for (uint64_t i = group_off[g]; i < group_off[g + 1]; i++) {
      poly_group[i] = g;
      chunk_off[i + 1] = chunk_off[i] + (uint32_t)((coeff_off[i + 1] - coeff_off[i] + KZG_OPEN_CH - 1) / KZG_OPEN_CH);
    }
  for (uint32_t i = 0; i < n_polys; i++) for (uint32_t b = chunk_off[i]; b < chunk_off[i + 1]; b++) chunk_poly.push_back(i);
  // k_kzg_eval_chunks
  std::vector<Fr255> agg(chunk_poly.size());
  for (uint32_t b = 0; b < chunk_poly.size(); b++) {
    const uint32_t p = chunk_poly[b];
    const uint32_t len = (uint32_t)(coeff_off[p + 1] - coeff_off[p]);
    const uint8_t* a = coeffs + 32 * coeff_off[p];
    const Fr255 z = load_mont(zs + (size_t)32 * poly_group[p]);
    KzgSpan s[KZG_OPEN_THREADS];
    for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) {
      const uint32_t base = (b - chunk_off[p]) * KZG_OPEN_CH + KZG_OPEN_SEG * t;
      s[t] = {kzg_segment_value(z, [&](int m) { return base + m < len ? load_mont(a + (size_t)32 * (base + m)) : Fr255::zero(); }),
              kzg_pow2k(z, KZG_OPEN_LOG_SEG)};
    }
    for (unsigned d = 1; d < 32; d <<= 1) {            // __shfl_down_sync: every lane reads lane + d (itself past the warp) first
      KzgSpan up[KZG_OPEN_THREADS];
      for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) up[t] = (t & 31u) + d < 32 ? s[t + d] : s[t];
      for (uint32_t t = 0; t < KZG_OPEN_THREADS; t++) s[t] = kzg_span_combine(s[t], up[t]);
    }
    KzgSpan c = s[0];
    for (int u = 1; u < KZG_OPEN_THREADS / 32; u++) c = kzg_span_combine(c, s[32 * u]);
    agg[b] = c.h;
  }
  // k_kzg_eval_finish
  for (uint32_t i = 0; i < n_polys; i++) {
    const Fr255 z_ch = kzg_pow2k(load_mont(zs + (size_t)32 * poly_group[i]), KZG_OPEN_LOG_CH);
    const Fr255* A = agg.data() + chunk_off[i];
    store_canonical(out_values + (size_t)32 * i, kzg_chunk_horner(z_ch, chunk_off[i + 1] - chunk_off[i], [&](uint32_t c) { return A[c]; }));
  }
  // k_kzg_aggregate, one group at a time
  for (uint32_t g = 0; g < n_groups; g++) {
    const uint32_t len = (uint32_t)(row_off[g + 1] - row_off[g]);
    uint8_t* row = out_rows + 32 * row_off[g];
    for (uint32_t base = 0; base < len; base += KZG_OPEN_SEG) {
      Fr255 acc[KZG_OPEN_SEG];
      for (int m = 0; m < KZG_OPEN_SEG; m++) acc[m] = Fr255::zero();
      for (uint64_t i = group_off[g]; i < group_off[g + 1]; i++) {
        const uint32_t len_i = (uint32_t)(coeff_off[i + 1] - coeff_off[i]);
        if (base >= len_i) continue;
        const Fr255 nu = load_mont(nus + (size_t)32 * i);
        const uint8_t* a = coeffs + 32 * (coeff_off[i] + base);
        for (int m = 0; m < KZG_OPEN_SEG; m++)
          if (base + m < len_i) acc[m] = acc[m] + kzg_agg_term(nu, load_reduced(a + 32 * m));
      }
      for (int m = 0; m < KZG_OPEN_SEG; m++)
        if (base + m < len) store_le<8>(row + (size_t)32 * (base + m), acc[m].v);
    }
  }
}
