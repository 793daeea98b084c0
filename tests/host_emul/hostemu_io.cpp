// TEST INFRASTRUCTURE ONLY: the item function of the prepared-input kernel (lincomb.cuh lincomb_io_item, V = s*I_j - c*O)
// compiled for the HOST, over input tables built by the same functions as on the GPU (key_table_powers / key_table_window).
// Built by tests/test_host_emul_prepared_io.py into a temporary directory; nothing in the product links this file.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../../ark_ec_vrfs_b200/csrc/gen/field_consts.cuh"
#include "../../ark_ec_vrfs_b200/csrc/lincomb.cuh"
using namespace vrfs;

// tables of n_in input points (n_in x 64 bytes); returns the key_ok flags of key_table_powers in ok[]
template <class C> static std::vector<typename Grp<C>::FixEntry> input_tables(int n_in, const uint8_t* pts, uint8_t* ok) {
  std::vector<typename Grp<C>::FixEntry> t((size_t)n_in * key_table_entries<C>());
  for (int j = 0; j < n_in; j++) {
    ok[j] = key_table_powers<C>(&t[(size_t)j * key_table_entries<C>()], pts + 64 * j);
    for (int w = 0; w < fix_windows<C, KEY_FIX_BITS>(); w++) key_table_window<C>(&t[(size_t)j * key_table_entries<C>() + (size_t)w * KEY_ENTRIES]);
  }
  return t;
}

// R = (-1)^(neg & 1) c*O + (-1)^(neg >> 1 & 1) s*I_j over the tables of n_in inputs, affine canonical out (x||y LE); returns
// lincomb_io_item's flag (O canonical and on the curve) | the table flags of the inputs in bits 1..n_in
template <class C> static int io_dbg(int n_in, const uint8_t* inputs, uint32_t j, const uint8_t* s, const uint8_t* o, const uint8_t* c,
                                     uint32_t c_bits, int neg_mask, uint8_t* out) {
  std::vector<uint8_t> tok(n_in);
  const auto tables = input_tables<C>(n_in, inputs, tok.data());
  std::vector<typename Grp<C>::Entry> slab(2 * TBL_ENTRIES);
  IoArgs A = {};
  A.L.n = 1;
  A.L.var[0] = {o, 64, c, 32, (uint32_t)(neg_mask & 1), c_bits};
  A.L.fix[0] = {s, 32, (uint32_t)((neg_mask >> 1) & 1), tables.data()};
  A.input_index = &j;
  A.n_inputs = (uint32_t)n_in;
  typename Grp<C>::Pt acc;
  int flags = lincomb_io_item<C>(A, 0, slab.data(), acc) ? 1 : 0;
  for (int i = 0; i < n_in; i++) flags |= tok[i] << (1 + i);
  alignas(16) uint32_t xyz[24];
  Grp<C>::store_xyz(xyz, acc);
  typename C::F X, Y, Z;
  memcpy(X.v, xyz, 32); memcpy(Y.v, xyz + 8, 32); memcpy(Z.v, xyz + 16, 32);
  typename C::F zi = inv(Z), x = X * zi, y = Y * zi;
  uint32_t rx[8], ry[8]; from_mont<typename C::Fq>(rx, x); from_mont<typename C::Fq>(ry, y);
  store_le<8>(out, rx); store_le<8>(out + 32, ry);
  return flags;
}
extern "C" int hostemu_lincomb_io(int suite, int n_in, const uint8_t* inputs, uint32_t j, const uint8_t* s, const uint8_t* o, const uint8_t* c,
                                  uint32_t c_bits, int neg_mask, uint8_t* out) {
  return suite == 0 ? io_dbg<BandCurve>(n_in, inputs, j, s, o, c, c_bits, neg_mask, out)
       : suite == 1 ? io_dbg<EdCurve>(n_in, inputs, j, s, o, c, c_bits, neg_mask, out) : io_dbg<P256Curve>(n_in, inputs, j, s, o, c, c_bits, neg_mask, out);
}
