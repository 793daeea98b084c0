// PreparedPublics::from_compressed / verify_signatures of include/vrfs_b200.hpp: serialised signatures of 7 signers published as
// encoded keys, verified by key index, give the verdicts, hashes and errors of Public::verify_signatures on the gathered encodings;
// a damaged signature, a wrong key and an index out of range fail on their own item only, and a bad key encoding has key_ok = 0.
#include <algorithm>
#include <cstdio>
#include <string>

#include "../../include/vrfs_b200.hpp"

using namespace vrfs;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); failures++; } } while (0)

int main() {
  const size_t n_keys = 7, n = 50;
  Engine eng(0);
  Suite suite = Suite::bandersnatch(eng);
  const size_t L = suite.point_enc_len(), hl = suite.hash_len();
  std::vector<Bytes> seeds, datas, ad;
  for (size_t k = 0; k < n_keys; k++) { std::string t = "wire-signer-" + std::to_string(k); seeds.push_back(Bytes(t.begin(), t.end())); }
  Secret keys = Secret::from_seed(suite, seeds);
  Bytes enc = keys.public_().serialize_compressed();
  enc.resize(L * (n_keys + 1), 0xFF);                       // key 7: not a canonical encoding
  std::vector<uint32_t> index(n);
  Bytes sk(32 * n);
  for (size_t i = 0; i < n; i++) {
    index[i] = (uint32_t)((i * 5 + 3) % n_keys);
    std::copy_n(keys.scalars.begin() + 32 * index[i], 32, sk.begin() + 32 * i);
    std::string t = "prepared-wire-" + std::to_string(i);
    datas.push_back(Bytes(t.begin(), t.end()));
    ad.push_back(Bytes(i % 5, (uint8_t)i));
  }
  Packed d(datas), a(ad);
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(suite.id);
  Bytes sigs(n * sl), sok(n);
  eng.check(vrfs_ietf_sign_wire_batch(eng.ctx(), suite.id, n, sk.data(), d.ptr(), d.off.data(), a.ptr(), a.off.data(), sigs.data(), sok.data()));
  for (size_t i = 0; i < n; i++) CHECK(sok[i] == 1);

  PreparedPublics prepared = PreparedPublics::from_compressed(suite, enc);
  CHECK(prepared.size() == n_keys + 1);
  for (size_t k = 0; k < n_keys; k++) CHECK(prepared.key_ok()[k] == 1);
  CHECK(prepared.key_ok()[n_keys] == 0);
  Errors errs;
  auto [ok, beta] = prepared.verify_signatures(index, datas, sigs, ad, &errs);
  for (size_t i = 0; i < n; i++) CHECK(ok[i] == 1 && errs[i] == Error::None);

  sigs[sl * 20 + L] ^= 1;                                   // a damaged challenge
  index[33] = (uint32_t)((index[33] + 1) % n_keys);         // a valid but wrong key
  index[40] = (uint32_t)n_keys;                             // the key that did not decode
  index[49] = (uint32_t)n_keys + 1;                         // out of range
  auto [ok1, beta1] = prepared.verify_signatures(index, datas, sigs, ad, &errs);
  Bytes gathered(n * L);
  for (size_t i = 0; i < n; i++) std::copy_n(enc.begin() + L * std::min<size_t>(index[i], n_keys), L, gathered.begin() + L * i);
  Errors errs_w;
  auto [ok_w, beta_w] = Public::verify_signatures(suite, gathered, datas, sigs, ad, &errs_w);
  for (size_t i = 0; i < n - 1; i++) CHECK(ok1[i] == ok_w[i] && errs[i] == errs_w[i]);
  CHECK(std::equal(beta1.begin(), beta1.begin() + hl * (n - 1), beta_w.begin()));
  for (size_t i = 0; i < n; i++) CHECK(ok1[i] == (i != 20 && i != 33 && i != 40 && i != 49));
  CHECK(errs[20] == Error::VerificationFailure && errs[33] == Error::VerificationFailure && errs[40] == Error::InvalidData &&
        errs[49] == Error::InvalidData);
  CHECK(std::all_of(beta1.begin() + hl * 49, beta1.end(), [](uint8_t b) { return b == 0; }));
  CHECK(std::equal(beta1.begin(), beta1.begin() + hl, beta.begin()));

  if (failures) return 1;
  std::printf("all ok\n");
  return 0;
}
